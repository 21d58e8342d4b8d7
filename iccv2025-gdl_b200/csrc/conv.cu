// conv.cu — implicit-GEMM convolution forward / dgrad / wgrad for sm_100a.
//
// Replaces the cuDNN convolutions the reference reaches through nn.Conv2d
// (reference models/backbone.py:20-28 conv3x3/conv1x1, :97-100 stems; backward through
// autograd from main_dgl.py:110,122).  Activations are NHWC bf16, accumulation is fp32 in
// TMEM, MMAs are tcgen05.mma (kind::f16, M=128) issued by a single thread.
//
//   fwd / dgrad : D[128 pixels, BN out-ch] = A[pixels, K] * W[out-ch, K]^T      (both K-major)
//        A rows are gathered on the fly (im2col never materialised): for k-block kb the
//        row of pixel m is 64 contiguous channels of one filter tap (or, for the 8-channel
//        padded stems, 8 taps x 8 channels), zero-filled outside the image.
//   wgrad       : D[(tap,ci) 128, BN co] = X_shift[pixels, (tap,ci)]^T * dY[pixels, co]
//        both operands MN-major (the reduction dimension is the pixel index), split-K over
//        pixel ranges with fp32 partials reduced in a fixed order (deterministic).
//
// All tiles live in shared memory in the 128-byte-swizzled canonical layout (row = 128 B,
// 16-byte chunk c of row r at chunk c^(r&7)), written by cp.async with zero-fill and made
// visible to the tensor core with fence.proxy.async before the mbarrier arrive.
#include <stdlib.h>
#include "common.cuh"
#include "tc05.cuh"

namespace gdl {
using namespace tc05;

struct ConvParams {
  const bf16* src;  // gathered tensor [N,Hs,Ws,Cs]
  const bf16* wt;   // [Cd][K] bf16, K-major
  bf16* dst;        // [N,Hd,Wd,Cd]
  const bf16* add_src;
  int add_mode, Hc, Wc;
  int N, Hs, Ws, Cs, Hd, Wd, Cd;
  int R, S, stride, pad;
  int mode;   // 0: hs = hd*stride + r - pad (forward); 1: hs = (hd + pad - r)/stride (dgrad)
  int ch8;    // 1: Cs == 8, a k-block is 8 taps x 8 channels
  int cshift; // log2(Cs/64) when !ch8
  int M, KB, K;
};

struct WgradParams {
  const bf16* x;   // gathered tensor [N,Hs,Ws,Cs]
  const bf16* dy;  // [N,Hd,Wd,Cd]
  float* partial;  // [splits][Kp][Cd]
  int N, Hs, Ws, Cs, Hd, Wd, Cd;
  int R, S, stride, pad;
  int ch8, cshift;
  int M;       // N*Hd*Wd (reduction length)
  int NAB;     // number of 64-wide A blocks = Kp/64
  int num_mt;  // ceil(NAB/2) 128-row M tiles
  int G;       // M tiles per CTA
  int kb_total, kb_per_split, Kp;
};

// Resolve which source pixel feeds (dst pixel, tap) and whether it is inside the image.
struct TapGeom {
  int R, S, stride, pad, mode, Hs, Ws;
};
__device__ __forceinline__ bool tap_source(const TapGeom& g, int hd, int wd, int tap, int& hs,
                                           int& ws) {
  if (tap >= g.R * g.S) return false;
  int r = tap / g.S;
  int s = tap - r * g.S;
  if (g.mode == 0) {
    hs = hd * g.stride + r - g.pad;
    ws = wd * g.stride + s - g.pad;
  } else {
    int nh = hd + g.pad - r, nw = wd + g.pad - s;
    if (nh < 0 || nw < 0) return false;
    hs = nh / g.stride;
    ws = nw / g.stride;
    if (hs * g.stride != nh || ws * g.stride != nw) return false;
  }
  return hs >= 0 && hs < g.Hs && ws >= 0 && ws < g.Ws;
}

// One 128-byte swizzled row of a gathered block.  ab = index of the 64-wide K block.
__device__ __forceinline__ void gather_row(const bf16* __restrict__ src, const TapGeom& g, int Cs,
                                           int ch8, int cshift, uint32_t blk_smem, int row,
                                           bool pix_valid, int n, int hd, int wd, int ab) {
  const uint32_t row_base = blk_smem + row * 128;
  const int sw = row & 7;
  if (!ch8) {
    int tap = ab >> cshift;
    int cb = ab - (tap << cshift);
    int hs = 0, ws = 0;
    bool valid = pix_valid && tap_source(g, hd, wd, tap, hs, ws);
    const bf16* p = valid ? src + ((size_t)((size_t)n * g.Hs + hs) * g.Ws + ws) * Cs + cb * 64 : src;
    uint32_t bytes = valid ? 16u : 0u;
#pragma unroll
    for (int c = 0; c < 8; ++c) cp_async16(row_base + ((c ^ sw) << 4), p + c * 8, bytes);
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      int hs = 0, ws = 0;
      bool valid = pix_valid && tap_source(g, hd, wd, ab * 8 + j, hs, ws);
      const bf16* p = valid ? src + ((size_t)((size_t)n * g.Hs + hs) * g.Ws + ws) * 8 : src;
      cp_async16(row_base + ((j ^ sw) << 4), p, valid ? 16u : 0u);
    }
  }
}

// ------------------------------------------------------------------------------------------
// forward / dgrad kernel: one 128 x BN output tile per CTA, 5 warps:
//   warps 0-3: cp.async producers during the main loop, then the TMEM epilogue
//   warp 4   : TMEM allocation + the single MMA-issuing thread
// ------------------------------------------------------------------------------------------
constexpr int kProducerThreads = 128;
constexpr int kConvThreads = 160;
constexpr int kLag = 2;  // cp.async groups kept in flight per producer thread

template <int BN, int STAGES>
struct ConvSmem {
  static constexpr int A_BYTES = 128 * 128;
  static constexpr int B_BYTES = BN * 128;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int BAR_OFF = STAGES * STAGE_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;  // barriers + alignment slack
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(kConvThreads) conv_igemm_kernel(const __grid_constant__ ConvParams p) {
  using L = ConvSmem<BN, STAGES>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* empty = full + STAGES;
  uint64_t* tmem_full = empty + STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int m0 = blockIdx.x * 128;
  const int n0 = blockIdx.y * BN;

  if (tid == 0) {
    for (int i = 0; i < STAGES; ++i) {
      mbar_init(&full[i], kProducerThreads);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, BN);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);

  if (warp < 4) {
    // ------------------------------ producers ------------------------------
    const int row = tid;  // A row == output pixel of the tile; also B row (weights) if < BN
    const int m = m0 + row;
    const bool pix_valid = m < p.M;
    int n = 0, hd = 0, wd = 0;
    if (pix_valid) {
      n = m / (p.Hd * p.Wd);
      int rem = m - n * p.Hd * p.Wd;
      hd = rem / p.Wd;
      wd = rem - hd * p.Wd;
    }
    TapGeom g{p.R, p.S, p.stride, p.pad, p.mode, p.Hs, p.Ws};
    const bf16* wrow = p.wt + (size_t)(n0 + (row < BN ? row : 0)) * p.K;
    const int sw = row & 7;

    for (int kb = 0; kb < p.KB; ++kb) {
      const int st = kb % STAGES;
      if (kb >= STAGES) mbar_wait(&empty[st], ((kb / STAGES) - 1) & 1);
      const uint32_t sA = smem_base + st * L::STAGE_BYTES;
      const uint32_t sB = sA + L::A_BYTES;
      gather_row(p.src, g, p.Cs, p.ch8, p.cshift, sA, row, pix_valid, n, hd, wd, kb);
      if (row < BN) {
        const bf16* w = wrow + kb * 64;
        const uint32_t rb = sB + row * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c) cp_async16(rb + ((c ^ sw) << 4), w + c * 8, 16u);
      }
      cp_async_commit();
      if (kb >= kLag) {
        cp_async_wait<kLag>();
        fence_proxy_async();
        mbar_arrive(&full[(kb - kLag) % STAGES]);
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    for (int kb = (p.KB > kLag ? p.KB - kLag : 0); kb < p.KB; ++kb) mbar_arrive(&full[kb % STAGES]);

    // ------------------------------ epilogue ------------------------------
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int lane = tid & 31;
    const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16);
    bf16* out = p.dst + (size_t)m * p.Cd + n0;
    const bf16* add = nullptr;
    if (pix_valid && p.add_mode == 1) {
      add = p.add_src + (size_t)m * p.Cd + n0;
    } else if (pix_valid && p.add_mode == 2) {
      if (((hd | wd) & 1) == 0)
        add = p.add_src + ((size_t)((size_t)n * p.Hc + (hd >> 1)) * p.Wc + (wd >> 1)) * p.Cd + n0;
    }
    (void)lane;
#pragma unroll 1
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      tmem_ld32(trow + c0, r);
      tmem_ld_wait();
      if (pix_valid) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[q * 8 + i]);
          if (add != nullptr) {
            float a[8];
            uint4 u = *reinterpret_cast<const uint4*>(add + c0 + q * 8);
            unpack8(u, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] += a[i];
          }
          *reinterpret_cast<uint4*>(out + c0 + q * 8) = pack8(f);
        }
      }
    }
  } else if (tid == kProducerThreads) {
    // ------------------------------ MMA issuer ------------------------------
    constexpr uint32_t idesc = make_idesc_bf16(128, BN, 0, 0);
    const uint32_t ab_hi = desc_hi_sw128(1024), ab_lo0 = desc_lo_sw128(smem_base, 16);
    for (int kb = 0; kb < p.KB; ++kb) {
      const int st = kb % STAGES;
      mbar_wait(&full[st], (kb / STAGES) & 1);
      tc_fence_after();
      const uint32_t a_lo = ab_lo0 + st * (L::STAGE_BYTES >> 4);
      const uint32_t b_lo = a_lo + (L::A_BYTES >> 4);
#pragma unroll
      for (int k = 0; k < 4; ++k)
        mma_bf16_ss(tmem_base, desc_join(a_lo + 2 * k, ab_hi), desc_join(b_lo + 2 * k, ab_hi), idesc,
                    (kb | k) != 0 ? 1u : 0u);
      mma_commit(&empty[st]);
    }
    mma_commit(tmem_full);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, BN);
}

// ------------------------------------------------------------------------------------------
// wgrad kernel: CTA (m-group, n-tile, split) accumulates G M-tiles x BN columns in TMEM over
// its pixel range; dY tile is loaded once per pixel block and reused by the G gathered tiles.
// ------------------------------------------------------------------------------------------
template <int BN, int AST>
struct WgradSmem {
  static constexpr int A_BYTES = 2 * 64 * 128;          // two 64-row blocks
  static constexpr int B_BYTES = (BN / 64) * 64 * 128;  // BN/64 blocks
  static constexpr int B_OFF = AST * A_BYTES;
  static constexpr int BAR_OFF = B_OFF + 2 * B_BYTES;
  static constexpr int TOTAL = BAR_OFF + 256 + 1024;
};

template <int BN, int AST>
__global__ void __launch_bounds__(kConvThreads) conv_wgrad_kernel(const __grid_constant__ WgradParams p) {
  using L = WgradSmem<BN, AST>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* a_full = reinterpret_cast<uint64_t*>(smem + L::BAR_OFF);
  uint64_t* a_empty = a_full + AST;
  uint64_t* b_full = a_empty + AST;
  uint64_t* b_empty = b_full + 2;
  uint64_t* tmem_full = b_empty + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);

  const int tid = threadIdx.x;
  const int warp = tid >> 5;
  const int mt0 = blockIdx.x * p.G;
  const int Gc = min(p.G, p.num_mt - mt0);
  const int n0 = blockIdx.y * BN;
  const int split = blockIdx.z;
  const int kb0 = split * p.kb_per_split;
  const int nkb = min(p.kb_per_split, p.kb_total - kb0);
  // TMEM columns: power of two >= 32 covering G*BN
  uint32_t ncols = 32;
  while (ncols < uint32_t(p.G * BN)) ncols <<= 1;

  if (tid == 0) {
    for (int i = 0; i < AST; ++i) {
      mbar_init(&a_full[i], kProducerThreads);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&b_full[i], kProducerThreads);
      mbar_init(&b_empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, ncols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);
  const int OPS = 1 + Gc;

  if (warp < 4) {
    // ------------------------------ producers ------------------------------
    const int blk = tid >> 6;  // which 64-row block this thread fills
    const int row = tid & 63;  // pixel row inside the pixel block
    const int sw = row & 7;
    TapGeom g{p.R, p.S, p.stride, p.pad, 0, p.Hs, p.Ws};
    int issued = 0;
    auto arrive_for = [&](int j) {
      int kbi = j / OPS, idx = j - kbi * OPS;
      if (idx == 0)
        mbar_arrive(&b_full[kbi & 1]);
      else
        mbar_arrive(&a_full[(kbi * Gc + idx - 1) % AST]);
    };
    for (int kbi = 0; kbi < nkb; ++kbi) {
      const int pix = (kb0 + kbi) * 64 + row;
      const bool pix_valid = pix < p.M;
      int n = 0, hd = 0, wd = 0;
      if (pix_valid) {
        n = pix / (p.Hd * p.Wd);
        int rem = pix - n * p.Hd * p.Wd;
        hd = rem / p.Wd;
        wd = rem - hd * p.Wd;
      }
      // dY tile: [64 pixels][BN co] as BN/64 blocks
      if (kbi >= 2) mbar_wait(&b_empty[kbi & 1], ((kbi >> 1) - 1) & 1);
      if (blk < BN / 64) {
        const bf16* s = pix_valid ? p.dy + (size_t)pix * p.Cd + n0 + blk * 64 : p.dy;
        const uint32_t rb = smem_base + L::B_OFF + (kbi & 1) * L::B_BYTES + blk * 8192 + row * 128;
        const uint32_t bytes = pix_valid ? 16u : 0u;
#pragma unroll
        for (int c = 0; c < 8; ++c) cp_async16(rb + ((c ^ sw) << 4), s + c * 8, bytes);
      }
      cp_async_commit();
      ++issued;
      if (issued > kLag) {
        cp_async_wait<kLag>();
        fence_proxy_async();
        arrive_for(issued - 1 - kLag);
      }
      for (int gi = 0; gi < Gc; ++gi) {
        const int ac = kbi * Gc + gi;
        const int st = ac % AST;
        if (ac >= AST) mbar_wait(&a_empty[st], ((ac / AST) - 1) & 1);
        const int ab = 2 * (mt0 + gi) + blk;
        gather_row(p.x, g, p.Cs, p.ch8, p.cshift, smem_base + st * L::A_BYTES + blk * 8192, row,
                   pix_valid && ab < p.NAB, n, hd, wd, ab);
        cp_async_commit();
        ++issued;
        if (issued > kLag) {
          cp_async_wait<kLag>();
          fence_proxy_async();
          arrive_for(issued - 1 - kLag);
        }
      }
    }
    cp_async_wait<0>();
    fence_proxy_async();
    for (int j = (issued > kLag ? issued - kLag : 0); j < issued; ++j) arrive_for(j);

    // ------------------------------ epilogue ------------------------------
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int lane = tid & 31;
    const int drow = warp * 32 + lane;
    const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16);
    for (int gi = 0; gi < Gc; ++gi) {
      const int k = (mt0 + gi) * 128 + drow;
      float* out = p.partial + ((size_t)split * p.Kp + k) * p.Cd + n0;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(trow + gi * BN + c0, r);
        tmem_ld_wait();
        if (k < p.Kp) {
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(out + c0 + q * 4) =
                make_uint4(r[q * 4], r[q * 4 + 1], r[q * 4 + 2], r[q * 4 + 3]);
        }
      }
    }
  } else if (tid == kProducerThreads) {
    // ------------------------------ MMA issuer ------------------------------
    constexpr uint32_t idesc = make_idesc_bf16(128, BN, 1, 1);
    const uint32_t mn_hi = desc_hi_sw128(1024);
    const uint32_t a_lo0 = desc_lo_sw128(smem_base, 8192), b_lo0 = desc_lo_sw128(smem_base + L::B_OFF, 8192);
    for (int kbi = 0; kbi < nkb; ++kbi) {
      mbar_wait(&b_full[kbi & 1], (kbi >> 1) & 1);
      tc_fence_after();
      const uint32_t b_lo = b_lo0 + (kbi & 1) * (L::B_BYTES >> 4);
      for (int gi = 0; gi < Gc; ++gi) {
        const int ac = kbi * Gc + gi;
        const int st = ac % AST;
        mbar_wait(&a_full[st], (ac / AST) & 1);
        tc_fence_after();
        const uint32_t a_lo = a_lo0 + st * (L::A_BYTES >> 4);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          mma_bf16_ss(tmem_base + gi * BN, desc_join(a_lo + k * (2048 >> 4), mn_hi),
                      desc_join(b_lo + k * (2048 >> 4), mn_hi), idesc, (kbi | k) != 0 ? 1u : 0u);
        mma_commit(&a_empty[st]);
      }
      mma_commit(&b_empty[kbi & 1]);
    }
    mma_commit(tmem_full);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, ncols);
}

// ------------------------------------------------------------------------------------------
// small helper kernels: weight packing, split-K reduction
// ------------------------------------------------------------------------------------------
__global__ void pack_weights_kernel(const float* __restrict__ w, bf16* __restrict__ wp,
                                    bf16* __restrict__ wT, int Co, int Ci, int ci_real, int R,
                                    int S, int Kp, int ch8) {
  // one thread per packed element (co, k)
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)Co * Kp) return;
  int co = int(idx / Kp), k = int(idx - (int64_t)co * Kp);
  int tap = k / Ci, ci = k - tap * Ci;
  (void)ch8;
  float v = 0.f;
  bool valid = tap < R * S && ci < ci_real;
  if (valid) {
    int r = tap / S, s = tap - r * S;
    v = w[(((size_t)co * ci_real + ci) * R + r) * S + s];
  }
  bf16 b = __float2bfloat16_rn(v);
  wp[idx] = b;
  if (wT != nullptr && valid) wT[(size_t)ci * (R * S * Co) + (size_t)tap * Co + co] = b;
}

// Multi-tensor variant: one launch refreshes the bf16 shadows of a whole encoder (reference
// main_dgl.py:154 optimizer.step() is followed by nothing — the shadows are this library's own state).
__global__ void pack_weights_multi_kernel(const gdl_pack_entry* __restrict__ tab, int n, int64_t total) {
  for (int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (int64_t)gridDim.x * blockDim.x) {
    int lo = 0, hi = n - 1;  // last entry with start <= idx
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tab[mid].start <= idx) lo = mid; else hi = mid - 1;
    }
    const gdl_pack_entry e = tab[lo];
    const int64_t li = idx - e.start;
    const int co = int(li / e.Kp), k = int(li - (int64_t)co * e.Kp);
    const int tap = k / e.Ci, ci = k - tap * e.Ci;
    float v = 0.f;
    const bool valid = tap < e.R * e.S && ci < e.ci_real;
    if (valid) {
      const int r = tap / e.S, s2 = tap - r * e.S;
      v = e.w[(((size_t)co * e.ci_real + ci) * e.R + r) * e.S + s2];
      if (e.scale != nullptr) v *= e.scale[co];  // eval mode: BatchNorm scale folded into the weights
    }
    const bf16 b = __float2bfloat16_rn(v);
    reinterpret_cast<bf16*>(e.wp)[li] = b;
    if (e.wT != nullptr && valid)
      reinterpret_cast<bf16*>(e.wT)[(size_t)ci * (e.R * e.S * e.Co) + (size_t)tap * e.Co + co] = b;
  }
}

// Tiled variant for the block convolutions (Ci % 64 == 0, Co % 32 == 0, no channel padding): the element-wise kernel
// above reads the OIHW master with a 36-byte stride per lane and scatters the transposed shadow in 2-byte pieces
// (0.15 ms per encoder for 11 M weights).  Here one CTA moves a [32 co][64 ci][R*S] tile through shared memory:
// coalesced fp32 reads (64*R*S contiguous floats per co), 128-byte runs into wp[co][tap][ci], 64-byte runs into
// wT[ci][tap][co].  blockIdx.y = table entry, blockIdx.x = tile (CTAs beyond the entry's tile count exit).
__global__ void __launch_bounds__(256) pack_weights_tiled_kernel(const gdl_pack_entry* __restrict__ tab) {
  extern __shared__ bf16 s_tile[];  // [32 co][RS][64 ci + 2 pad] (row stride 33 words: the transposed read is conflict-free)
  constexpr int LD = 66;
  const gdl_pack_entry e = tab[blockIdx.y];
  const int RS = e.R * e.S;
  const int ci_tiles = e.Ci >> 6, tiles = (e.Co >> 5) * ci_tiles;
  if ((int)blockIdx.x >= tiles) return;
  const int co0 = (blockIdx.x / ci_tiles) << 5, ci0 = (blockIdx.x % ci_tiles) << 6;
  const int run = 64 * RS;  // contiguous floats per output channel in the OIHW master
  for (int i = threadIdx.x; i < 32 * run; i += 256) {
    const int co = i / run, r = i - co * run;
    const int ci = r / RS, tap = r - ci * RS;
    float v = e.w[((size_t)(co0 + co) * e.Ci + ci0) * RS + r];
    if (e.scale != nullptr) v *= e.scale[co0 + co];
    s_tile[(co * RS + tap) * LD + ci] = __float2bfloat16_rn(v);
  }
  __syncthreads();
  bf16* wp = reinterpret_cast<bf16*>(e.wp);
  for (int i = threadIdx.x; i < 32 * run; i += 256) {  // wp[co][tap*Ci + ci]: 64 consecutive ci per (co, tap)
    const int ci = i & 63, ct = i >> 6, co = ct / RS, tap = ct - co * RS;
    wp[(size_t)(co0 + co) * e.Kp + (size_t)tap * e.Ci + ci0 + ci] = s_tile[ct * LD + ci];
  }
  if (e.wT != nullptr) {
    bf16* wT = reinterpret_cast<bf16*>(e.wT);
    for (int i = threadIdx.x; i < 32 * run; i += 256) {  // wT[ci][tap*Co + co]: 32 consecutive co per (ci, tap)
      const int co = i & 31, ct = i >> 5, tap = ct % RS, ci = ct / RS;
      wT[(size_t)(ci0 + ci) * (RS * e.Co) + (size_t)tap * e.Co + co0 + co] = s_tile[(co * RS + tap) * LD + ci];
    }
  }
}

__global__ void wgrad_reduce_kernel(const float* __restrict__ partial, float* __restrict__ dw,
                                    int splits, int Kp, int Cd, int Ci, int ci_real, int R, int S) {
  int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // (k, co), co fastest
  if (idx >= (int64_t)Kp * Cd) return;
  int k = int(idx / Cd), co = int(idx - (int64_t)k * Cd);
  int tap = k / Ci, ci = k - tap * Ci;
  if (tap >= R * S || ci >= ci_real) return;
  float acc = 0.f;
  for (int sp = 0; sp < splits; ++sp) acc += partial[(size_t)sp * Kp * Cd + idx];
  int r = tap / S, s = tap - r * S;
  dw[(((size_t)co * ci_real + ci) * R + r) * S + s] = acc;
}

// Split-K reduction of the flat weight-gradient kernel's CO-MAJOR partials [split][Co][Kp] into the fp32 OIHW
// gradient.  The split loop is the latency chain (one dependent add per split), so small weight tensors
// (64x64x9 = 36 k outputs, up to 148 splits) spread it over G thread groups: group g sums splits g, g+G, ...
// four loads in flight, and thread group 0 combines the G partial sums in ascending g — a fixed order, so the
// result is deterministic (reference utils.py:12 cudnn.deterministic).  Reads are coalesced over k = (tap, ci).
struct TapSplits {
  int n[9];  // splits that wrote tap t's partials (parity planes of a stride-2 conv get different counts)
};
template <int G>
__global__ void __launch_bounds__(256) wgrad_reduce_t_kernel(const float* __restrict__ partial, float* __restrict__ dw,
                                                             const TapSplits ts, int Kp, int Co, int Ci, int taps) {
  constexpr int OB = 256 / G;  // outputs per block
  __shared__ float red[G > 1 ? 256 : 1];
  const int o = threadIdx.x % OB, g = threadIdx.x / OB;
  const int64_t total = (int64_t)Co * Kp;
  const int64_t idx = (int64_t)blockIdx.x * OB + o;  // (co, k), k fastest
  float acc = 0.f;
  const int co = int(idx / Kp), k = int(idx - (int64_t)co * Kp);
  const int tap = k / Ci, ci = k - tap * Ci;
  if (idx < total) {
    const float* src = partial + idx;
    const int splits = ts.n[tap];
    int sp = g;
    for (; sp + 3 * G < splits; sp += 4 * G) {
      const float a0 = src[(size_t)sp * total], a1 = src[(size_t)(sp + G) * total];
      const float a2 = src[(size_t)(sp + 2 * G) * total], a3 = src[(size_t)(sp + 3 * G) * total];
      acc += a0;
      acc += a1;
      acc += a2;
      acc += a3;
    }
    for (; sp < splits; sp += G) acc += src[(size_t)sp * total];
  }
  if (G > 1) {
    red[threadIdx.x] = acc;
    __syncthreads();
    if (g != 0) return;
#pragma unroll
    for (int j = 1; j < G; ++j) acc += red[j * OB + o];
  }
  if (idx >= total) return;
  dw[((size_t)co * Ci + ci) * taps + tap] = acc;
}

static int launch_wgrad_reduce_t(const float* partial, float* dw, int splits, const TapSplits& ts, int Kp, int Co,
                                 int Ci, int taps, cudaStream_t s) {
  const int64_t total = (int64_t)Co * Kp;
  // (A shared-memory-transposing variant that writes contiguous OIHW runs was measured for the large layers and was
  // 2-5 % slower per weight gradient than the per-element kernel below: the partials are L2-resident and the
  // 36-byte-stride stores of 2.4 M elements do not bound it.)
  if (total < 400000 && splits >= 16) {
    wgrad_reduce_t_kernel<8><<<(unsigned)ceil_div64(total, 32), 256, 0, s>>>(partial, dw, ts, Kp, Co, Ci, taps);
  } else if (total < 800000 && splits >= 8) {
    wgrad_reduce_t_kernel<4><<<(unsigned)ceil_div64(total, 64), 256, 0, s>>>(partial, dw, ts, Kp, Co, Ci, taps);
  } else {
    wgrad_reduce_t_kernel<1><<<(unsigned)ceil_div64(total, 256), 256, 0, s>>>(partial, dw, ts, Kp, Co, Ci, taps);
  }
  GDL_CHECK_LAUNCH("wgrad_reduce_t_kernel");
  return GDL_OK;
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

static bool desc_ok(const gdl_conv_desc* d) {
  if (!d) return false;
  if (d->N <= 0 || d->Hi <= 0 || d->Wi <= 0 || d->Ho <= 0 || d->Wo <= 0) return false;
  if (!(d->Ci == 8 || (d->Ci % 64 == 0 && (d->Ci & (d->Ci - 1)) == 0))) return false;
  if (d->Co % 64 != 0) return false;
  if (d->R <= 0 || d->S <= 0 || d->stride <= 0 || d->pad < 0) return false;
  if ((int64_t)d->N * d->Ho * d->Wo >= (int64_t)1 << 31) return false;
  if ((int64_t)d->N * d->Hi * d->Wi >= (int64_t)1 << 31) return false;
  return true;
}

static int packed_k(const gdl_conv_desc* d) { return (d->R * d->S * d->Ci + 63) / 64 * 64; }

struct WgradPlan {
  int BN, G, NAB, num_mt, mgroups, ntiles, kb_total, kb_per_split, splits, Kp;
};
static WgradPlan plan_wgrad(const gdl_conv_desc* d) {
  WgradPlan w;
  w.Kp = packed_k(d);
  w.BN = d->Co == 64 ? 64 : 128;
  w.NAB = w.Kp / 64;
  w.num_mt = (w.NAB + 1) / 2;
  int gmax = 512 / w.BN;
  if (gmax > 4) gmax = 4;
  w.G = w.num_mt < gmax ? w.num_mt : gmax;
  // balance: 5 M-tiles with gmax 4 would give groups of 4+1; prefer 3+2
  w.mgroups = (w.num_mt + w.G - 1) / w.G;
  w.G = (w.num_mt + w.mgroups - 1) / w.mgroups;
  w.ntiles = d->Co / w.BN;
  int64_t M = (int64_t)d->N * d->Ho * d->Wo;
  w.kb_total = int((M + 63) / 64);
  int target = 2 * kNumSMs;
  int splits = target / (w.mgroups * w.ntiles);
  if (splits < 1) splits = 1;
  if (splits > w.kb_total) splits = w.kb_total;
  w.kb_per_split = (w.kb_total + splits - 1) / splits;
  w.splits = (w.kb_total + w.kb_per_split - 1) / w.kb_per_split;
  return w;
}

template <int BN, int STAGES>
static int launch_igemm(const ConvParams& p, cudaStream_t s) {
  using L = ConvSmem<BN, STAGES>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_igemm_kernel<BN, STAGES>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(conv_igemm)");
    attr_set = true;
  }
  dim3 grid((p.M + 127) / 128, p.Cd / BN);
  conv_igemm_kernel<BN, STAGES><<<grid, kConvThreads, L::TOTAL, s>>>(p);
  GDL_CHECK_LAUNCH("conv_igemm_kernel");
  return GDL_OK;
}

template <int BN, int AST>
static int launch_wgrad(const WgradParams& p, const WgradPlan& w, cudaStream_t s) {
  using L = WgradSmem<BN, AST>;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel<BN, AST>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(conv_wgrad)");
    attr_set = true;
  }
  dim3 grid(w.mgroups, w.ntiles, w.splits);
  conv_wgrad_kernel<BN, AST><<<grid, kConvThreads, L::TOTAL, s>>>(p);
  GDL_CHECK_LAUNCH("conv_wgrad_kernel");
  return GDL_OK;
}

// conv_flat.cu
int try_conv_flat(int kind, int N, int Hs, int Ws, int Cs, int64_t sW, int64_t sH, int64_t sN, const void* src,
                  const void* wt, int64_t wt_rows, int64_t wt_k, void* dst, int Hd, int Wd, int Cd,
                  const void* add_src, int add_mode, cudaStream_t s, float* stats = nullptr,
                  int* stats_rows = nullptr, const float* bias = nullptr, int relu = 0);

// GDL_FLAT=0 routes every convolution to the generic gather kernels below (conv_igemm_kernel / conv_wgrad_kernel:
// cp.async im2col gather, any geometry) instead of the flat-window TMA kernels — the fallback for geometries the flat
// kernels do not cover (rows wider than 255 pixels, channel counts that are not multiples of 64), exercised by
// tests/test_gpu_kernels.py::test_generic_gather_kernels.  Default: flat wherever eligible.
static int flat_policy() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("GDL_FLAT");
    v = e ? atoi(e) : 2;
  }
  return v;
}
// 1x1 convolutions up to this many input channels take the flat kernel (round 1 stopped at 128: the 256 -> 512
// downsample of layer4 ran on the legacy gather kernel at 8 % tensor-pipe activity)
constexpr int kFlat1x1MaxCi = 512;
static bool prefer_flat_s1(int, int) { return flat_policy() != 0; }

// conv_wgrad_flat.cu
int64_t wgrad_flat_workspace_bytes(int N, int Ho, int Wo, int Ci, int Co, int R, int stride);
int try_wgrad_flat(int N, int Hi, int Wi, int Ho, int Wo, int Ci, int Co, int R, int stride, const void* x,
                   const void* dy, float* partial, int64_t workspace_bytes, cudaStream_t s, int transposed,
                   int* tap_splits);
// GDL_WFLAT=0: generic gather weight-gradient kernel instead of the flat-window one (see GDL_FLAT above)
static int wflat_policy() {
  static int v = -1;
  if (v < 0) {
    const char* e = getenv("GDL_WFLAT");
    v = e ? atoi(e) : 2;
  }
  return v;
}
static bool wflat_shape_ok(const gdl_conv_desc* d) {
  if (d->Ci % 64 != 0 || d->R != d->S) return false;
  if (d->R == 3) return d->pad == 1 && (d->stride == 1 || d->stride == 2);
  return d->R == 1 && d->pad == 0 && (d->stride == 1 || d->stride == 2);
}
static bool prefer_wflat(const gdl_conv_desc* d) { return wflat_policy() != 0 && wflat_shape_ok(d); }

static int run_igemm(const ConvParams& p, cudaStream_t s) {
  if (p.Cd % 128 == 0) return launch_igemm<128, 3>(p, s);
  return launch_igemm<64, 4>(p, s);
}

}  // namespace gdl

using namespace gdl;

extern "C" int64_t gdl_conv_packed_k(const gdl_conv_desc* d) { return desc_ok(d) ? packed_k(d) : GDL_EINVAL; }

extern "C" int64_t gdl_conv_wgrad_workspace_bytes(const gdl_conv_desc* d) {
  if (!desc_ok(d)) return GDL_EINVAL;
  WgradPlan w = plan_wgrad(d);
  int64_t need = (int64_t)w.splits * w.Kp * d->Co * (int64_t)sizeof(float);
  if (wflat_shape_ok(d)) {
    int64_t f = wgrad_flat_workspace_bytes(d->N, d->Ho, d->Wo, d->Ci, d->Co, d->R, d->stride);
    if (f > need) need = f;
  }
  return need;
}

extern "C" int gdl_conv_pack_weights(const gdl_conv_desc* d, int ci_real, const float* w_oihw,
                                     void* w_packed, void* w_packed_T, gdl_stream_t s) {
  GDL_REQUIRE(desc_ok(d), "gdl_conv_pack_weights: bad descriptor");
  GDL_REQUIRE(w_oihw && w_packed, "gdl_conv_pack_weights: null pointer");
  GDL_REQUIRE(ci_real > 0 && ci_real <= d->Ci, "gdl_conv_pack_weights: ci_real out of range");
  GDL_REQUIRE(w_packed_T == nullptr || d->Ci % 64 == 0, "gdl_conv_pack_weights: no transposed pack for stems");
  int Kp = packed_k(d);
  int64_t total = (int64_t)d->Co * Kp;
  pack_weights_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)s>>>(
      w_oihw, (bf16*)w_packed, (bf16*)w_packed_T, d->Co, d->Ci, ci_real, d->R, d->S, Kp, d->Ci == 8);
  GDL_CHECK_LAUNCH("pack_weights_kernel");
  return GDL_OK;
}

// bias / res / relu: eval-mode epilogue y = [relu](conv + bias[co] [+ res]) (gdl_conv_fwd_bias_act); flat kernels only
static int conv_fwd_impl(const gdl_conv_desc* d, const void* x, const void* w_packed, void* y, float* stats,
                         int* stats_rows, gdl_stream_t s, const float* bias = nullptr, const void* res = nullptr,
                         int relu = 0) {
  const bool epi = bias != nullptr || res != nullptr || relu != 0;
  const int amode = res != nullptr ? 1 : 0;
  GDL_REQUIRE(desc_ok(d), "gdl_conv_fwd: bad descriptor");
  GDL_REQUIRE(x && w_packed && y, "gdl_conv_fwd: null pointer");
  if (stats_rows) *stats_rows = 0;
  if (d->R == 3 && d->S == 3 && d->stride == 1 && d->pad == 1 && d->Ci % 64 == 0) {
    if (prefer_flat_s1(d->Hi, d->Wi) || epi) {
      int rc = try_conv_flat(0, d->N, d->Hi, d->Wi, d->Ci, d->Ci, (int64_t)d->Wi * d->Ci,
                             (int64_t)d->Hi * d->Wi * d->Ci, x, w_packed, d->Co, 9 * (int64_t)d->Ci, y, d->Ho, d->Wo,
                             d->Co, res, amode, (cudaStream_t)s, stats, stats_rows, bias, relu);
      if (rc != 0) return rc < 0 ? rc : GDL_OK;
    }
  }
  if (d->R == 3 && d->S == 3 && d->stride == 2 && d->pad == 1 && d->Ci % 64 == 0 && flat_policy() != 0) {
    // stride 2: the four parity planes of x are stride-1 sources on the output grid
    int rc = try_conv_flat(4, d->N, d->Ho, d->Wo, d->Ci, d->Ci, (int64_t)d->Wi * d->Ci,
                           (int64_t)d->Hi * d->Wi * d->Ci, x, w_packed, d->Co, 9 * (int64_t)d->Ci, y, d->Ho, d->Wo,
                           d->Co, res, amode, (cudaStream_t)s, stats, stats_rows, bias, relu);
    if (rc != 0) return rc < 0 ? rc : GDL_OK;
  }
  if (d->R == 1 && d->S == 1 && d->pad == 0 && d->Ci % 64 == 0 && d->Ci <= kFlat1x1MaxCi && flat_policy() != 0) {
    // 1x1 (stride 1 or 2): a single tap over the strided view x[:, ::stride, ::stride, :]
    int rc = try_conv_flat(3, d->N, d->Ho, d->Wo, d->Ci, (int64_t)d->stride * d->Ci,
                           (int64_t)d->stride * d->Wi * d->Ci, (int64_t)d->Hi * d->Wi * d->Ci, x, w_packed, d->Co,
                           (int64_t)d->Ci, y, d->Ho, d->Wo, d->Co, res, amode, (cudaStream_t)s, stats, stats_rows, bias,
                           relu);
    if (rc != 0) return rc < 0 ? rc : GDL_OK;
  }
  if (epi) {
    set_last_error("gdl_conv_fwd_bias_act: this geometry is not covered by the flat-window kernels");
    return GDL_EINVAL;
  }
  ConvParams p{};
  p.src = (const bf16*)x;
  p.wt = (const bf16*)w_packed;
  p.dst = (bf16*)y;
  p.add_src = nullptr;
  p.add_mode = 0;
  p.N = d->N; p.Hs = d->Hi; p.Ws = d->Wi; p.Cs = d->Ci;
  p.Hd = d->Ho; p.Wd = d->Wo; p.Cd = d->Co;
  p.R = d->R; p.S = d->S; p.stride = d->stride; p.pad = d->pad;
  p.mode = 0;
  p.ch8 = d->Ci == 8;
  p.cshift = p.ch8 ? 0 : ilog2(d->Ci / 64);
  p.M = d->N * d->Ho * d->Wo;
  p.K = packed_k(d);
  p.KB = p.K / 64;
  return run_igemm(p, (cudaStream_t)s);
}

extern "C" int gdl_conv_pack_weights_tiled(const gdl_pack_entry* table_dev, int n, int max_tiles, int max_rs,
                                           gdl_stream_t s) {
  GDL_REQUIRE(table_dev && n > 0 && max_tiles > 0 && max_rs > 0 && max_rs <= 9, "gdl_conv_pack_weights_tiled: bad arguments");
  const size_t smem = (size_t)32 * max_rs * 66 * sizeof(bf16);
  pack_weights_tiled_kernel<<<dim3(max_tiles, n), 256, smem, (cudaStream_t)s>>>(table_dev);
  GDL_CHECK_LAUNCH("pack_weights_tiled_kernel");
  return GDL_OK;
}

extern "C" int gdl_conv_pack_weights_multi(const gdl_pack_entry* table_dev, int n, int64_t total, gdl_stream_t s) {
  GDL_REQUIRE(table_dev && n > 0 && total > 0, "gdl_conv_pack_weights_multi: bad arguments");
  int64_t blocks = ceil_div64(total, 256);
  if (blocks > kNumSMs * 8) blocks = kNumSMs * 8;
  pack_weights_multi_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)s>>>(table_dev, n, total);
  GDL_CHECK_LAUNCH("pack_weights_multi_kernel");
  return GDL_OK;
}

extern "C" int gdl_conv_fwd(const gdl_conv_desc* d, const void* x, const void* w_packed, void* y,
                            gdl_stream_t s) {
  return conv_fwd_impl(d, x, w_packed, y, nullptr, nullptr, s);
}

extern "C" int gdl_conv_fwd_bias_act(const gdl_conv_desc* d, const void* x, const void* w_packed, const float* bias,
                                     const void* res, int relu, void* y, gdl_stream_t s) {
  GDL_REQUIRE(bias != nullptr, "gdl_conv_fwd_bias_act: null bias");
  return conv_fwd_impl(d, x, w_packed, y, nullptr, nullptr, s, bias, res, relu ? 1 : 0);
}

extern "C" int gdl_conv_fwd_stats(const gdl_conv_desc* d, const void* x, const void* w_packed, void* y,
                                  float* bn_partial, int* bn_partial_rows, gdl_stream_t s) {
  GDL_REQUIRE(bn_partial && bn_partial_rows, "gdl_conv_fwd_stats: null pointer");
  return conv_fwd_impl(d, x, w_packed, y, bn_partial, bn_partial_rows, s);
}

extern "C" int gdl_conv_dgrad(const gdl_conv_desc* d, const void* dy, const void* w_packed_T,
                              void* dx, const void* add_src, int add_mode, gdl_stream_t s) {
  GDL_REQUIRE(desc_ok(d), "gdl_conv_dgrad: bad descriptor");
  GDL_REQUIRE(d->Ci % 64 == 0, "gdl_conv_dgrad: stems have no data gradient");
  GDL_REQUIRE(dy && w_packed_T && dx, "gdl_conv_dgrad: null pointer");
  GDL_REQUIRE(add_mode >= 0 && add_mode <= 2 && (add_mode == 0 || add_src), "gdl_conv_dgrad: bad add_mode");
  if (d->R == 3 && d->S == 3 && d->stride == 1 && d->pad == 1) {
    if (prefer_flat_s1(d->Hi, d->Wi) && add_mode != 2) {
      int rc = try_conv_flat(1, d->N, d->Ho, d->Wo, d->Co, d->Co, (int64_t)d->Wo * d->Co,
                             (int64_t)d->Ho * d->Wo * d->Co, dy, w_packed_T, d->Ci, 9 * (int64_t)d->Co, dx, d->Hi,
                             d->Wi, d->Ci, add_src, add_mode, (cudaStream_t)s);
      if (rc != 0) return rc < 0 ? rc : GDL_OK;
    }
  }
  if (d->R == 3 && d->S == 3 && d->stride == 2 && d->pad == 1 && add_mode != 1 && flat_policy() != 0) {
    // four output-parity classes, 1+2+2+4 taps instead of 9 zero-stuffed ones
    int rc = try_conv_flat(2, d->N, d->Ho, d->Wo, d->Co, d->Co, (int64_t)d->Wo * d->Co,
                           (int64_t)d->Ho * d->Wo * d->Co, dy, w_packed_T, d->Ci, 9 * (int64_t)d->Co, dx, d->Hi,
                           d->Wi, d->Ci, add_src, add_mode, (cudaStream_t)s);
    if (rc != 0) return rc < 0 ? rc : GDL_OK;
  }
  if (d->R == 1 && d->S == 1 && d->stride == 1 && d->pad == 0 && add_mode != 2 && flat_policy() != 0) {
    int rc = try_conv_flat(3, d->N, d->Ho, d->Wo, d->Co, d->Co, (int64_t)d->Wo * d->Co,
                           (int64_t)d->Ho * d->Wo * d->Co, dy, w_packed_T, d->Ci, (int64_t)d->Co, dx, d->Hi, d->Wi,
                           d->Ci, add_src, add_mode, (cudaStream_t)s);
    if (rc != 0) return rc < 0 ? rc : GDL_OK;
  }
  ConvParams p{};
  p.src = (const bf16*)dy;
  p.wt = (const bf16*)w_packed_T;
  p.dst = (bf16*)dx;
  p.add_src = (const bf16*)add_src;
  p.add_mode = add_mode;
  p.Hc = (d->Hi + 1) / 2;
  p.Wc = (d->Wi + 1) / 2;
  p.N = d->N; p.Hs = d->Ho; p.Ws = d->Wo; p.Cs = d->Co;
  p.Hd = d->Hi; p.Wd = d->Wi; p.Cd = d->Ci;
  p.R = d->R; p.S = d->S; p.stride = d->stride; p.pad = d->pad;
  p.mode = 1;
  p.ch8 = 0;
  p.cshift = ilog2(d->Co / 64);
  GDL_REQUIRE((d->Co & (d->Co - 1)) == 0, "gdl_conv_dgrad: Co must be a power of two");
  p.M = d->N * d->Hi * d->Wi;
  p.K = d->R * d->S * d->Co;
  p.KB = p.K / 64;
  return run_igemm(p, (cudaStream_t)s);
}

extern "C" int gdl_conv_wgrad(const gdl_conv_desc* d, int ci_real, const void* x, const void* dy,
                              float* dw_oihw, void* workspace, int64_t workspace_bytes,
                              gdl_stream_t s) {
  GDL_REQUIRE(desc_ok(d), "gdl_conv_wgrad: bad descriptor");
  GDL_REQUIRE(x && dy && dw_oihw && workspace, "gdl_conv_wgrad: null pointer");
  GDL_REQUIRE(ci_real > 0 && ci_real <= d->Ci, "gdl_conv_wgrad: ci_real out of range");
  if (ci_real == d->Ci && prefer_wflat(d)) {
    // co-major partials (coalesced epilogue stores) + the group-parallel reduction
    TapSplits ts;
    for (int i = 0; i < 9; ++i) ts.n[i] = 0;
    int ns = try_wgrad_flat(d->N, d->Hi, d->Wi, d->Ho, d->Wo, d->Ci, d->Co, d->R, d->stride, x, dy, (float*)workspace,
                            workspace_bytes, (cudaStream_t)s, 1, ts.n);
    if (ns < 0) return ns;
    if (ns > 0)
      return launch_wgrad_reduce_t((const float*)workspace, dw_oihw, ns, ts, d->R * d->S * d->Ci, d->Co, d->Ci,
                                   d->R * d->S, (cudaStream_t)s);
  }
  WgradPlan w = plan_wgrad(d);
  int64_t need = (int64_t)w.splits * w.Kp * d->Co * (int64_t)sizeof(float);
  if (workspace_bytes < need) {
    set_last_error("gdl_conv_wgrad: workspace too small");
    return GDL_ENOMEM;
  }
  WgradParams p{};
  p.x = (const bf16*)x;
  p.dy = (const bf16*)dy;
  p.partial = (float*)workspace;
  p.N = d->N; p.Hs = d->Hi; p.Ws = d->Wi; p.Cs = d->Ci;
  p.Hd = d->Ho; p.Wd = d->Wo; p.Cd = d->Co;
  p.R = d->R; p.S = d->S; p.stride = d->stride; p.pad = d->pad;
  p.ch8 = d->Ci == 8;
  p.cshift = p.ch8 ? 0 : ilog2(d->Ci / 64);
  p.M = d->N * d->Ho * d->Wo;
  p.NAB = w.NAB; p.num_mt = w.num_mt; p.G = w.G;
  p.kb_total = w.kb_total; p.kb_per_split = w.kb_per_split; p.Kp = w.Kp;
  int rc = (w.BN == 128) ? launch_wgrad<128, 4>(p, w, (cudaStream_t)s)
                         : launch_wgrad<64, 4>(p, w, (cudaStream_t)s);
  if (rc != GDL_OK) return rc;
  int64_t total = (int64_t)w.Kp * d->Co;
  wgrad_reduce_kernel<<<(unsigned)ceil_div64(total, 256), 256, 0, (cudaStream_t)s>>>(
      (const float*)workspace, dw_oihw, w.splits, w.Kp, d->Co, d->Ci, ci_real, d->R, d->S);
  GDL_CHECK_LAUNCH("wgrad_reduce_kernel");
  return GDL_OK;
}
