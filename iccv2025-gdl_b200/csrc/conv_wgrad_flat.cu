// conv_wgrad_flat.cu — weight gradient on flat pixel windows (reference models/backbone.py:44,47,
// 142-145 conv3x3 / conv1x1 backward, reached from main_dgl.py:110):
//
//   dW[co][tap][ci] = sum over pixels   dY[pix][co] * X_plane(tap)[pix + (dr,dc)(tap)][ci]
//
// One pipeline stage is ONE TMA box per operand slab: either a band of RB full-width rows of one
// image, or (small maps) NI whole images.  Boxes are P = Wo+1 pixels wide — the extra column is TMA
// out-of-bounds zero fill and serves as the right pad of a row and the left pad of the next — and the
// X box starts rmin rows above the dY box, so inside shared memory pixel i of the dY window meets its
// tap (dr,dc) at X row i + (dr-rmin)*P + dc: a constant row shift, for every pixel of the stage.  Rows
// above/below an image are out-of-bounds zero fill as well; whole-image boxes are Ho+1 rows per image so
// that one zero row is both the bottom pad of image n and the top pad of image n+1.  Zero pixels (pads,
// rows past the image, the 16-row K-step tail) contribute nothing; the slack rows around the windows are
// zeroed once at kernel start and never written again.  7x7 maps fill 77 % of every K step (16x8 pixel
// tiles: 38 %), 14x14 87 %, 65x47 98 %.
//   Stride-2 convolutions read X through its four parity planes (strided tensor-map views on the
//   output grid): tap (r,s) lives in plane ((r+1)&1, (s+1)&1) at (dr,dc) = (r==0 ? -1 : 0, s==0 ? -1 : 0).
//   Both operands are MN-major (rows = pixels = the reduction dimension); D[(tap,ci) 128][BN co]
//   accumulates in TMEM over the CTA's stage range (split-K); fp32 partials are written once per CTA and
//   reduced in a fixed order (deterministic).
//   MODE 0 (Ci == 64): an M tile is TWO taps x 64 ci (second block = same window, LBO rows further).
//   MODE 1 (Ci >= 128): an M tile is one tap x 128 ci (two slab windows, LBO = slab stride).
#include <stdlib.h>
#include <string.h>
#include "common.cuh"
#include "tma.cuh"

namespace gdl {
using namespace tc05;

constexpr int kWfThreads = 192;
constexpr int kWfMaxUnits = 5;
constexpr int kWfMaxPx = 256;

struct WfUnit {
  int shift;       // X row of block 0 relative to the dY pixel, in the stage's row units
  int lbo;         // MODE 0: byte distance to the second tap's rows
  int tap0, tap1;  // linear tap indices (r*S+s) of the two 64-row blocks; tap1 < 0: unused block
};
struct WfJobType {
  int plane, nunits, rmin;
  WfUnit u[kWfMaxUnits];
};
struct WfParams {
  CUtensorMap tm_x[4];  // box {64, P, xrows, NI}
  CUtensorMap tm_dy;    // box {64, P, dyrows, NI}
  float* partial;       // [splits][Kp][Co], or [splits][Co][Kp] when transposed
  int transposed;       // 1: partials stored co-major, so a warp's 32 rows (consecutive ci) store 128 contiguous bytes
  int Ci, Co, Kp;
  int ntypes;
  WfJobType jt[4];
  int ci_tiles, co_tiles;
  int NI, RB, nbands;   // stage = NI whole images (nbands == 1, RB == Ho+1) or one RB-row band of one image
  int ksteps;           // ceil(stage pixels / 16)
  int tiles_total;
  int tps[4];           // tiles per split-K CTA of each job type (types with more taps get more, shorter, splits)
  int xwin_bytes, dywin_bytes, stage_bytes, stages;
  uint32_t tx_bytes;
  int smem_bytes;
};

template <int BN, int MODE>
__global__ void __launch_bounds__(kWfThreads, 1) conv_wgrad_flat_kernel(const __grid_constant__ WfParams p) {
  constexpr int NS = MODE == 0 ? 1 : 2;
  constexpr int NB = BN / 64;
  constexpr int kMaxSt = 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint64_t* full = reinterpret_cast<uint64_t*>(smem + p.stages * p.stage_bytes);
  uint64_t* empty = full + kMaxSt;
  uint64_t* tmem_full = empty + kMaxSt;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full + 1);
  const int tid = threadIdx.x, warp = warp_uniform_idx();
  const int ST = p.stages;
  int y = blockIdx.y;
  const int type = y % p.ntypes;
  const int t0 = min(blockIdx.x * p.tps[type], p.tiles_total);
  const int t1 = min(t0 + p.tps[type], p.tiles_total);
  if (t0 >= t1) return;  // this type has fewer splits than the grid is wide (whole CTA, before any setup)
  y /= p.ntypes;
  const int co0 = (y % p.co_tiles) * BN;
  const int ci0 = (y / p.co_tiles) * (NS * 64);
  const WfJobType& jt = p.jt[type];

  // zero the stage buffers once: the slack rows around the TMA boxes must read as zero forever
  {
    uint4* z = reinterpret_cast<uint4*>(smem);
    const int n16 = (p.stages * p.stage_bytes) >> 4;
    for (int i = tid; i < n16; i += kWfThreads) z[i] = make_uint4(0, 0, 0, 0);
  }
  if (tid == 0) {
    for (int i = 0; i < kMaxSt; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(tmem_full, 1);
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  if (tid == 5 * 32) {
    tma_prefetch_desc(&p.tm_x[jt.plane]);
    tma_prefetch_desc(&p.tm_dy);
  }
  fence_proxy_async();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);
  const int dy_off = NS * p.xwin_bytes;

  if (warp == 5 && elect_one()) {
    // ------------------------------ TMA producer ------------------------------
    const CUtensorMap* tmx = &p.tm_x[jt.plane];
    int it = 0;
    for (int t = t0; t < t1; ++t, ++it) {
      int n0, h0;
      if (p.nbands == 1) {
        n0 = t * p.NI;
        h0 = 0;
      } else {
        n0 = t / p.nbands;
        h0 = (t - n0 * p.nbands) * p.RB;
      }
      const int st = it % ST;
      if (it >= ST) mbar_wait(&empty[st], ((it / ST) - 1) & 1);
      mbar_arrive_expect_tx(&full[st], p.tx_bytes);
      const uint32_t sbase = smem_base + st * p.stage_bytes;
#pragma unroll
      for (int sl = 0; sl < NS; ++sl)  // +128: one zero row in front of the X box
        tma_load_4d(sbase + sl * p.xwin_bytes + 128, tmx, &full[st], ci0 + sl * 64, 0, h0 + jt.rmin, n0);
#pragma unroll
      for (int b = 0; b < NB; ++b)
        tma_load_4d(sbase + dy_off + b * p.dywin_bytes, &p.tm_dy, &full[st], co0 + b * 64, 0, h0, n0);
    }
  } else if (warp == 4 && elect_one()) {
    // ------------------------------ MMA issuer ------------------------------
    // One thread issues every MMA and is instruction-latency bound: all operands stay in uniform registers
    // (the kernel owns all 512 TMEM columns, so the base is column 0 — checked), the unit loop is unrolled
    // per unit count, and only the very first K step carries the "overwrite" predicate.
    if (tmem_base != 0) {
      printf("gdl: conv_wgrad_flat expects TMEM base 0, got %u\n", tmem_base);
      __trap();
    }
    constexpr uint32_t idesc = make_idesc_bf16(128, BN, 1, 1);
    const uint32_t hi = desc_hi_sw128(1024);  // 8-pixel K groups are dense rows in both windows
    // per-unit descriptor constants: (row shift + 1 front row) in 16-byte units, LBO in bits 16+
    uint32_t ua[kWfMaxUnits];
#pragma unroll
    for (int u = 0; u < kWfMaxUnits; ++u) {
      const uint32_t lbo = MODE == 0 ? (uint32_t)jt.u[u].lbo : (uint32_t)p.xwin_bytes;
      ua[u] = (uint32_t)((jt.u[u].shift + 1) * 8) + (((lbo >> 4) & 0x3FFFu) << 16);
    }
    const uint32_t ub = ((uint32_t)(p.dywin_bytes >> 4) & 0x3FFFu) << 16;
    const int nunits = jt.nunits;
    const int ksteps = p.ksteps;
    int it = 0;
    for (int t = t0; t < t1; ++t, ++it) {
      const int st = it % ST;
      mbar_wait(&full[st], (it / ST) & 1);
      tc_fence_after();
      const uint32_t sa = ((smem_base + st * p.stage_bytes) & 0x3FFFFu) >> 4;
      const uint32_t sb = sa + (dy_off >> 4) + ub;
      int j0 = 0;
      if (it == 0) {  // first K step of the CTA overwrites the accumulators
#pragma unroll
        for (int u = 0; u < kWfMaxUnits; ++u)
          if (u < nunits) mma_bf16_ss(u * BN, desc_join(sa + ua[u], hi), desc_join(sb, hi), idesc, 0u);
        j0 = 1;
      }
#define WF_ISSUE(NU)                                                                                          \
  for (int j = j0; j < ksteps; ++j) {                                                                         \
    const uint32_t b_lo = sb + j * 128;                                                                       \
    _Pragma("unroll") for (int u = 0; u < NU; ++u)                                                            \
        mma_bf16_acc(u * BN, desc_join(sa + ua[u] + j * 128, hi), desc_join(b_lo, hi), idesc);                \
  }
      switch (nunits) {
        case 1: WF_ISSUE(1) break;
        case 2: WF_ISSUE(2) break;
        case 3: WF_ISSUE(3) break;
        case 4: WF_ISSUE(4) break;
        default: WF_ISSUE(5) break;
      }
#undef WF_ISSUE
      mma_commit(&empty[st]);
    }
    mma_commit(tmem_full);
  } else if (warp < 4) {
    // ------------------------------ epilogue: fp32 partials ------------------------------
    mbar_wait(tmem_full, 0);
    tc_fence_after();
    const int row = tid;
    const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16);
#pragma unroll 1
    for (int u = 0; u < jt.nunits; ++u) {
      int tap, ci;
      if (MODE == 0) {
        tap = row < 64 ? jt.u[u].tap0 : jt.u[u].tap1;
        ci = row & 63;
      } else {
        tap = jt.u[u].tap0;
        ci = ci0 + row;
      }
      const bool valid = tap >= 0 && t1 > t0;
      const size_t krow = (size_t)(tap < 0 ? 0 : tap) * p.Ci + ci;
      // transposed: lane l of a warp owns row ci0+l, so for one output column the warp writes 32 consecutive
      // floats (one 128-byte line per store instruction); row-major partials put every lane on its own line
      // (32 lines per store instruction, i.e. 32x the LSU wavefronts for the same bytes).
      float* out = p.transposed ? p.partial + ((size_t)blockIdx.x * p.Co + co0) * p.Kp + krow
                                : p.partial + ((size_t)blockIdx.x * p.Kp + krow) * p.Co + co0;
#pragma unroll 1
      for (int c0 = 0; c0 < BN; c0 += 32) {
        uint32_t r[32];
        tmem_ld32(trow + u * BN + c0, r);
        tmem_ld_wait();
        if (valid) {
          if (p.transposed) {
#pragma unroll
            for (int i = 0; i < 32; ++i) out[(size_t)(c0 + i) * p.Kp] = __uint_as_float(r[i]);
          } else {
#pragma unroll
            for (int g = 0; g < 8; ++g)
              *reinterpret_cast<uint4*>(out + c0 + g * 4) = make_uint4(r[g * 4], r[g * 4 + 1], r[g * 4 + 2], r[g * 4 + 3]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 512);
}

// (A CTA-pair variant of this kernel — tcgen05.mma.cta_group::2, the two CTAs of a cluster on neighbouring ci tiles of
// one job, each holding half of the dY window — was written and validated in round 2 (Ci >= 256 layers) and measured
// at +2-5 % per weight gradient against this kernel on every layer of the bench geometry (14x14 C256: 0.198 vs 0.190 ms,
// 7x7 C512: 0.222 vs 0.217 ms): halving the dY operand traffic does not pay here, the weight gradient is not
// shared-memory or L2 bound the way the forward / data-gradient kernels are.  Removed again.)

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
struct WfPlan {
  int mode, BN, ntypes, ci_tiles, co_tiles, gy, splits, tiles_total;
  int tps[4], nsplit[4];  // per job type: tiles per CTA, number of split-K CTAs (splits = max nsplit)
  int xwin_bytes, dywin_bytes, stage_bytes, stages, P, taps;
  int NI, RB, nbands, ksteps, xrows, dyrows, rspan;
  WfJobType jt[4];
};

struct WfTap {
  int tap, plane, dr, dc;
};

static void wf_add_unit(WfJobType& t, int P, const WfTap& a, const WfTap* b) {
  WfUnit& u = t.u[t.nunits++];
  u.shift = (a.dr - t.rmin) * P + a.dc;
  u.tap0 = a.tap;
  u.tap1 = b ? b->tap : -1;
  u.lbo = b ? (((b->dr - t.rmin) * P + b->dc) - u.shift) * 128 : 128;
}

// R in {1,3}, stride in {1,2}; (Ho, Wo) is the output grid the pixel windows run over.
static bool plan_wgrad_flat(int N, int Ho, int Wo, int Ci, int Co, int R, int stride, WfPlan& w) {
  if (Ci % 64 != 0 || Co % 64 != 0) return false;
  if (!(R == 3 || R == 1) || !(stride == 1 || stride == 2)) return false;
  memset(&w, 0, sizeof(w));
  const int P = Wo + 1;
  if (P > 256) return false;
  w.P = P;
  w.taps = R * R;
  if (Ci == 64) {
    w.mode = 0;
    w.BN = Co == 64 ? 64 : 128;
    w.ci_tiles = 1;
  } else if (Ci % 128 == 0 && Co % 128 == 0) {
    w.mode = 1;
    w.BN = 128;
    w.ci_tiles = Ci / 128;
  } else {
    return false;
  }
  w.co_tiles = Co / w.BN;
  // --- taps and the job types (taps sharing one X window) ---
  WfTap taps[9];
  int nt = 0;
  for (int r = 0; r < R; ++r)
    for (int s = 0; s < R; ++s) {
      WfTap t;
      t.tap = r * R + s;
      if (R == 1) {
        t.plane = 0; t.dr = 0; t.dc = 0;
      } else if (stride == 1) {
        t.plane = 0; t.dr = r - 1; t.dc = s - 1;
      } else {
        t.plane = ((r + 1) & 1) * 2 + ((s + 1) & 1);
        t.dr = r == 0 ? -1 : 0;
        t.dc = s == 0 ? -1 : 0;
      }
      taps[nt++] = t;
    }
  w.rspan = 0;
  if (stride == 1 && w.mode == 1 && R == 3) {
    w.ntypes = 3;  // one filter row per CTA: 3 accumulators, narrow window
    for (int r = 0; r < 3; ++r) {
      w.jt[r].plane = 0;
      w.jt[r].rmin = r - 1;
      for (int s = 0; s < 3; ++s) wf_add_unit(w.jt[r], P, taps[r * 3 + s], nullptr);
    }
  } else {
    const int nplanes = (stride == 2 && R == 3) ? 4 : 1;
    for (int pl = 0; pl < nplanes; ++pl) {
      WfTap g[9];
      int ng = 0, rmin = 9, rmax = -9;
      for (int i = 0; i < nt; ++i)
        if (taps[i].plane == pl) {
          g[ng++] = taps[i];
          if (taps[i].dr < rmin) rmin = taps[i].dr;
          if (taps[i].dr > rmax) rmax = taps[i].dr;
        }
      if (ng == 0) continue;
      WfJobType& jt = w.jt[w.ntypes++];
      jt.plane = pl;
      jt.rmin = rmin;
      if (rmax - rmin > w.rspan) w.rspan = rmax - rmin;
      if (w.mode == 0) {
        for (int i = 0; i < ng; i += 2) wf_add_unit(jt, P, g[i], i + 1 < ng ? &g[i + 1] : nullptr);
      } else {
        for (int i = 0; i < ng; ++i) wf_add_unit(jt, P, g[i], nullptr);
      }
    }
  }
  for (int k = 0; k < w.ntypes; ++k) {
    if (w.jt[k].nunits * w.BN > 512) return false;
    for (int i = 0; i < w.jt[k].nunits; ++i)
      if (w.mode == 0 && w.jt[k].u[i].lbo <= 0) return false;
  }
  // --- stage geometry: NI whole images, or a band of RB rows; minimise K steps (+ per-stage overhead) ---
  const int NS = w.mode == 0 ? 1 : 2, NB = w.BN / 64;
  const int budget = 227 * 1024 - 2048;
  double best = 1e30;
  for (int whole = 0; whole < 2; ++whole) {
    for (int v = 1; v <= (whole ? 8 : Ho); whole ? v *= 2 : ++v) {
      const int NI = whole ? v : 1, RB = whole ? Ho + 1 : v;
      if (whole && w.rspan > 1) continue;
      const int px = NI * RB * P;
      if (px > kWfMaxPx) break;
      const int xrows = whole ? RB : RB + w.rspan;
      const int ks = (px + 15) / 16;
      // X window: 1 zero row + box + tail reachable by the largest shift from the last K step
      const int xwin = ((1 + ks * 16 + (w.rspan + 1) * P + 2) * 128 + 1023) / 1024 * 1024;
      const int xbox = NI * xrows * P * 128;
      if (xbox + 128 > xwin) continue;
      const int dywin = (ks * 16 * 128 + 1023) / 1024 * 1024;
      const int stage = NS * xwin + NB * dywin;
      int stages = budget / stage;
      if (stages > 4) stages = 4;
      if (stages < 2) continue;
      const int nb = whole ? 1 : (Ho + RB - 1) / RB;
      const int64_t tiles = whole ? (N + NI - 1) / NI : (int64_t)N * nb;
      double cost = (double)tiles * (ks + 1.5) * (stages >= 3 ? 1.0 : 1.25);
      if (cost < best) {
        best = cost;
        w.NI = NI; w.RB = RB; w.nbands = nb; w.ksteps = ks;
        w.xrows = xrows; w.dyrows = RB;
        w.xwin_bytes = xwin; w.dywin_bytes = dywin; w.stage_bytes = stage; w.stages = stages;
        w.tiles_total = (int)tiles;
      }
    }
  }
  if (best >= 1e30) return false;
  if (w.xwin_bytes >= (1 << 18) || w.dywin_bytes >= (1 << 18)) return false;  // LBO field
  w.gy = w.ci_tiles * w.co_tiles * w.ntypes;
  // One CTA per SM (the stage ring takes ~200 KB) and all 512 TMEM columns: CTAs of a second wave cannot
  // overlap the first wave's epilogue, they only add a prologue, an epilogue and a set of partials each: the
  // split-K factor is sized for one wave.
  // Split-K CTAs per job type, proportional to the type's MMA work per tile (its accumulator count): the
  // parity planes of a stride-2 convolution carry 4 / 2 / 2 / 1 taps, and with equal splits the 1-tap CTAs
  // would idle for 3/4 of the kernel.
  const int groups = w.ci_tiles * w.co_tiles;
  int cta_budget = kNumSMs / groups;  // CTAs of one (ci, co) tile over all types
  if (cta_budget < w.ntypes) cta_budget = w.ntypes;
  int wsum = 0;
  for (int k = 0; k < w.ntypes; ++k) wsum += w.jt[k].nunits;
  int used = 0;
  for (int k = 0; k < w.ntypes; ++k) {
    int sk = cta_budget * w.jt[k].nunits / wsum;
    if (sk < 1) sk = 1;
    w.nsplit[k] = sk;
    used += sk;
  }
  while (used < cta_budget) {  // hand the remainder to the type with the most work per CTA
    int best_k = 0;
    for (int k = 1; k < w.ntypes; ++k)
      if ((int64_t)w.jt[k].nunits * w.nsplit[best_k] > (int64_t)w.jt[best_k].nunits * w.nsplit[k]) best_k = k;
    ++w.nsplit[best_k];
    ++used;
  }
  w.splits = 0;
  for (int k = 0; k < w.ntypes; ++k) {
    int sk = w.nsplit[k] > w.tiles_total ? w.tiles_total : w.nsplit[k];
    w.tps[k] = (w.tiles_total + sk - 1) / sk;
    w.nsplit[k] = (w.tiles_total + w.tps[k] - 1) / w.tps[k];
    if (w.nsplit[k] > w.splits) w.splits = w.nsplit[k];
  }
  return true;
}

template <int BN, int MODE>
static int launch_wf(const WfParams& p, const WfPlan& w, cudaStream_t s) {
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_flat_kernel<BN, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         227 * 1024);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(conv_wgrad_flat)");
    attr_set = true;
  }
  dim3 grid(w.splits, w.gy);
  conv_wgrad_flat_kernel<BN, MODE><<<grid, kWfThreads, w.stages * w.stage_bytes + 512 + 1024, s>>>(p);
  GDL_CHECK_LAUNCH("conv_wgrad_flat_kernel");
  return GDL_OK;
}

// Workspace (bytes) the flat path needs, or 0 when the shape is not eligible.
int64_t wgrad_flat_workspace_bytes(int N, int Ho, int Wo, int Ci, int Co, int R, int stride) {
  WfPlan w;
  if (!plan_wgrad_flat(N, Ho, Wo, Ci, Co, R, stride, w)) return 0;
  return (int64_t)w.splits * w.taps * Ci * Co * (int64_t)sizeof(float);
}

// x is the conv INPUT [N,Hi,Wi,Ci]; dy the output gradient [N,Ho,Wo,Co].  Returns the number of splits
// written (>0) when handled, 0 when not eligible, <0 on error.
// transposed != 0: partials are written [split][Co][Kp] (coalesced epilogue stores), else [split][Kp][Co].
// tap_splits (optional, R*R ints): how many splits wrote each tap's partials (taps of different parity planes
// may have different split counts; the return value is the maximum).
int try_wgrad_flat(int N, int Hi, int Wi, int Ho, int Wo, int Ci, int Co, int R, int stride, const void* x,
                   const void* dy, float* partial, int64_t workspace_bytes, cudaStream_t s, int transposed,
                   int* tap_splits) {
  WfPlan w;
  if (!plan_wgrad_flat(N, Ho, Wo, Ci, Co, R, stride, w)) return 0;
  if (workspace_bytes < (int64_t)w.splits * w.taps * Ci * Co * (int64_t)sizeof(float)) return 0;
  WfParams p;
  memset(&p, 0, sizeof(p));
  const bf16* xb = (const bf16*)x;
  const int64_t sW = (int64_t)stride * Ci, sH = (int64_t)stride * Wi * Ci, sN = (int64_t)Hi * Wi * Ci;
  if (stride == 2 && R == 3) {
    // plane (a,b)[i,j] = x[2i+a, 2j+b]; its extent on the output grid is what exists of the input
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        const int ph = (Hi - a + 1) / 2, pw = (Wi - b + 1) / 2;
        if (ph <= 0 || pw <= 0) return 0;
        const CUtensorMap* t =
            tmap_view4(xb + ((int64_t)a * Wi + b) * Ci, Ci, pw, ph, N, sW, sH, sN, w.P, w.xrows, w.NI);
        if (!t) return GDL_ECUDA;
        p.tm_x[a * 2 + b] = *t;
      }
  } else {
    const CUtensorMap* t = tmap_view4(xb, Ci, Wo, Ho, N, sW, sH, sN, w.P, w.xrows, w.NI);
    if (!t) return GDL_ECUDA;
    p.tm_x[0] = *t;
  }
  const CUtensorMap* td =
      tmap_view4(dy, Co, Wo, Ho, N, Co, (int64_t)Wo * Co, (int64_t)Ho * Wo * Co, w.P, w.dyrows, w.NI);
  if (!td) return GDL_ECUDA;
  p.tm_dy = *td;
  p.partial = partial;
  p.transposed = transposed != 0;
  p.Ci = Ci; p.Co = Co; p.Kp = w.taps * Ci;
  p.ntypes = w.ntypes;
  for (int i = 0; i < 4; ++i) p.jt[i] = w.jt[i];
  p.ci_tiles = w.ci_tiles; p.co_tiles = w.co_tiles;
  p.NI = w.NI; p.RB = w.RB; p.nbands = w.nbands; p.ksteps = w.ksteps;
  p.tiles_total = w.tiles_total;
  for (int k = 0; k < 4; ++k) p.tps[k] = w.tps[k];
  if (tap_splits != nullptr)
    for (int k = 0; k < w.ntypes; ++k)
      for (int u = 0; u < w.jt[k].nunits; ++u) {
        tap_splits[w.jt[k].u[u].tap0] = w.nsplit[k];
        if (w.jt[k].u[u].tap1 >= 0) tap_splits[w.jt[k].u[u].tap1] = w.nsplit[k];
      }
  p.xwin_bytes = w.xwin_bytes; p.dywin_bytes = w.dywin_bytes; p.stage_bytes = w.stage_bytes; p.stages = w.stages;
  const int NS = w.mode == 0 ? 1 : 2, NB = w.BN / 64;
  p.tx_bytes = (uint32_t)((NS * w.xrows + NB * w.dyrows) * w.NI * w.P * 128);
  int rc;
  if (w.mode == 0)
    rc = w.BN == 64 ? launch_wf<64, 0>(p, w, s) : launch_wf<128, 0>(p, w, s);
  else
    rc = launch_wf<128, 1>(p, w, s);
  return rc == GDL_OK ? w.splits : rc;
}

}  // namespace gdl
