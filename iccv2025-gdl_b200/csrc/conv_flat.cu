// conv_flat.cu — "flat window" TMA implicit GEMM for every convolution whose taps are pure
// shifts on ONE pixel grid: 3x3/s1 forward and data-gradient at any map size (reference
// models/backbone.py:44,47 conv3x3), the data-gradient of the 3x3/s2 convolutions
// (backbone.py:44 with stride 2, split into its four output-parity classes so that only the
// structurally non-zero taps are multiplied), the 1x1/s2 downsample forward (backbone.py:142-145,
// through a strided tensor-map view) and the 1x1 data-gradient on the compact grid.
//
// The source grid [N,Hs,Ws] is indexed by ONE flat pixel index with a single zero pad column and
// a single zero pad row per image:
//        q = n*IS + h*P + w,   P = Ws+1,  IS = (Hs+1)*P,   h in [0,Hs], w in [0,Ws]
// (w == Ws is the pad column shared by the right edge of row h and the left edge of row h+1; h == Hs
// is the pad row shared by image n's bottom and image n+1's top).  A filter tap (dh,dw) is then the
// constant row shift dh*P+dw, for every pixel, across row and image boundaries.  An output tile is
// 128 (or 2x128) CONSECUTIVE q; its operand window [q0+smin, q0+M+smax) is brought into shared memory
// by one TMA box per padded row ({64 ch, P px}: the pad column/row are TMA out-of-bounds zero fill),
// and each tap's A operand is a row-shifted view of that window (the tensor core, like TMA, swizzles on
// absolute shared-memory address bits, so starts offset by whole 128-byte rows need no re-layout).
// Utilisation is Hs*Ws/((Hs+1)(Ws+1)) for every map size — 77 % at 7x7 and 9x6 where 16x8 pixel tiles
// reach 38-42 % — and the input is fetched from L2 once per 64-channel slab instead of once per tap.
//   warp 5 lane 0 : TMA producer (window ring + weight ring)
//   warp 4 lane 0 : tcgen05.mma issuer; MT accumulators share every weight tile
//   warps 0-3     : epilogue (TMEM -> registers -> bf16 NHWC, optional residual add), double-buffered
#include <string.h>
#include "common.cuh"
#include "tma.cuh"

namespace gdl {
using namespace tc05;

constexpr int kFlatThreads = 192;
constexpr int kFlatMaxTaps = 9;
constexpr int kFlatSmemBudget = 227 * 1024 - 2048;
constexpr int kFlatSmemFloor = 200 * 1024;

struct FlatTap {
  int shift;  // row shift on the flat grid (may be negative)
  int wk;     // k offset of the tap's weight columns in the packed matrix
};

struct FlatParams {
  CUtensorMap tm_x[4];  // {Cs, Ws, Hs, N} views of the source (one per parity plane), box {64, P, 1, 1}
  CUtensorMap tm_x4[4];    // same views, box {64, P, 4, 1}: four padded rows of one image per TMA operation
  CUtensorMap tm_ximg[4];  // same views, box {64, P, Hs+1, 1}: a whole padded image (small maps; see use_img)
  int use_r4, use_img;
  CUtensorMap tm_w;  // {K, rows} packed weights, box {64, BN}
  CUtensorMap tm_w_half;  // CTA-pair kernel: box {64, BN/2} (each CTA of a pair holds one half of every weight tile)
  bf16* dst;
  const bf16* add_src;
  float* stats;  // optional [gridDim.x * 4 epilogue warps][2][Cd]: per-warp sum / sum of squares of the bf16 outputs
  int add_mode;  // 0 none; 1 add_src has dst's shape; 2 add_src lives on the source grid (parity class (0,0) only)
  const float* bias;  // optional per-output-channel bias [Cd] (eval mode: the folded BatchNorm shift), added before relu
  int relu;           // eval-mode epilogue: clamp at zero after bias / residual
  int N, Hs, Ws, Cs;
  int Hd, Wd, Cd;
  int P, IS;
  int dscale;  // dst pixel = (h*dscale + ph, w*dscale + pw)
  int nclass;
  int ntaps[4];
  int ph[4], pw[4];
  FlatTap taps[4][kFlatMaxTaps];
  // taps of a class are ordered by group; a group = the taps that slide over ONE source view (plane)
  int ngroups[4];
  int gplane[4][4];
  int gtap0[4][5];  // group g of class c owns taps [gtap0[c][g], gtap0[c][g+1])
  int smin, smax;
  int mtiles, ntiles, items_total;
  int rev;  // gdl_set_sweep hint: walk the pixel tiles of every (class, channel tile) in descending order
  int res_tiles;  // RES kernels: number of weight tiles (taps x slabs) kept resident in shared memory
  int win_stage_bytes, win_stages;
};

__device__ __forceinline__ int floor_div(int a, int b) {  // b > 0
  int q = a / b;
  return (a - q * b < 0) ? q - 1 : q;
}

// ------------------------------------------------------------------------------------------
// BatchNorm statistics in the epilogue (reference backbone.py:45,48 train-mode BN over the conv output).
// An epilogue thread owns one pixel row of the tile, the statistics are per channel column: each warp transposes
// its 32 x 32 block of bf16-ROUNDED outputs (what BatchNorm will read; zero for pad rows) through a private
// 2.6 KB shared-memory scratch — lane l writes its row as four 16-byte vectors, then lane (hh, wd) reads the
// packed channel pair wd of rows hh*16 .. hh*16+15 — and accumulates sum / sum of squares in registers over all
// the CTA's tiles of one channel tile.  ~120 instructions per 32-column chunk (the shuffle butterfly this replaces
// needed ~350) and 4 KB of shared-memory traffic per chunk.  Row pitch 20 words, upper 16 rows displaced by 16
// words: row writes (8 lanes x 16 B per wavefront) and column reads (2 x 16 lanes x 4 B) are bank-conflict free.
// The order of every addition is fixed, so the statistics are deterministic.
constexpr int kStatRowBytes = 80;
constexpr int kStatWarpBytes = 32 * kStatRowBytes + 64;
constexpr int kStatScratchBytes = 4 * kStatWarpBytes;

template <int BN>
struct StatAcc {
  float s[BN / 32][2], q[BN / 32][2];
  int nt;
};

__device__ __forceinline__ void stat_chunk(uint32_t scratch, int lane, const uint4 (&o)[4], float (&s)[2],
                                           float (&q)[2]) {
  __syncwarp();  // the previous chunk's column reads are complete
  const uint32_t wrow = scratch + lane * kStatRowBytes + (lane >> 4) * 64;
#pragma unroll
  for (int v = 0; v < 4; ++v)
    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(wrow + v * 16), "r"(o[v].x), "r"(o[v].y), "r"(o[v].z),
                 "r"(o[v].w)
                 : "memory");
  __syncwarp();
  const uint32_t rcol = scratch + (lane >> 4) * (16 * kStatRowBytes + 64) + (lane & 15) * 4;
#pragma unroll
  for (int rr = 0; rr < 16; ++rr) {
    uint32_t w;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(rcol + rr * kStatRowBytes) : "memory");
    const float lo = __uint_as_float(w << 16), hi = __uint_as_float(w & 0xffff0000u);
    s[0] += lo;
    q[0] = fmaf(lo, lo, q[0]);
    s[1] += hi;
    q[1] = fmaf(hi, hi, q[1]);
  }
}

// Adds the warp's register sums of channel tile sa.nt into its private partial row [2][Cd] and clears them.
template <int BN>
__device__ __forceinline__ void stat_flush(StatAcc<BN>& sa, float* slot, int Cd, int lane) {
  if (slot == nullptr || sa.nt < 0) return;
  __syncwarp();
#pragma unroll
  for (int c = 0; c < BN / 32; ++c)
#pragma unroll
    for (int e = 0; e < 2; ++e) {
      const float s = sa.s[c][e] + __shfl_xor_sync(0xffffffffu, sa.s[c][e], 16);
      const float q = sa.q[c][e] + __shfl_xor_sync(0xffffffffu, sa.q[c][e], 16);
      if (lane < 16) {
        const int ch = sa.nt * BN + c * 32 + 2 * lane + e;
        slot[ch] += s;
        slot[Cd + ch] += q;
      }
      sa.s[c][e] = sa.q[c][e] = 0.f;
    }
}

// One item of the epilogue warps (shared by the single-CTA and the CTA-pair kernel): output addresses of this
// thread's MT pixel rows, residual prefetch, wait for the accumulator, TMEM -> registers -> bf16 NHWC.
// The residual rows (dgrad: gradient of the skip connection) are fetched into registers BEFORE the wait
// on the accumulator, one tile ahead, so their DRAM latency hides behind the MMAs instead of stalling the
// TMEM drain (measured: 0.45 -> 0.25 ms on the 56x56 C64 dgrads).
template <int BN, int MT, bool STATS>
__device__ __forceinline__ void flat_epilogue_item(const FlatParams& p, int cls, int n0, int q0, int tid, int lane,
                                                   uint64_t* full_bar, uint32_t full_parity, uint32_t trow,
                                                   uint32_t scratch, bool do_stats, StatAcc<BN>& sa) {
  constexpr int NV = BN / 8;  // 16-byte vectors per output row
  bf16* outp[MT];
  const bf16* addp[MT];
  bool validj[MT];
#pragma unroll
  for (int j = 0; j < MT; ++j) {
    const int q = q0 + j * 128 + tid;
    const int n = q / p.IS;
    const int r2 = q - n * p.IS;
    const int h = r2 / p.P, w = r2 - h * p.P;
    const int hd = h * p.dscale + p.ph[cls], wd = w * p.dscale + p.pw[cls];
    validj[j] = n < p.N && h < p.Hs && w < p.Ws && hd < p.Hd && wd < p.Wd;
    const size_t off = ((size_t)((size_t)n * p.Hd + hd) * p.Wd + wd) * p.Cd + n0;
    outp[j] = p.dst + off;
    addp[j] = nullptr;
    if (validj[j] && p.add_mode == 1)
      addp[j] = p.add_src + off;
    else if (validj[j] && p.add_mode == 2 && (p.ph[cls] | p.pw[cls]) == 0)
      addp[j] = p.add_src + ((size_t)((size_t)n * p.Hs + h) * p.Ws + w) * p.Cd + n0;
  }
  U32B res[NV / 2];
  const U32B zero32 = {make_uint4(0, 0, 0, 0), make_uint4(0, 0, 0, 0)};
  if (p.add_mode != 0) {
#pragma unroll
    for (int v = 0; v < NV / 2; ++v) res[v] = addp[0] ? ld_stream32(addp[0] + v * 16) : zero32;
  }
  mbar_wait(full_bar, full_parity);
  tc_fence_after();
#pragma unroll
  for (int j = 0; j < MT; ++j) {
    U32B nres[NV / 2];
    if (p.add_mode != 0 && j + 1 < MT) {  // next tile's residual row while this one drains
#pragma unroll
      for (int v = 0; v < NV / 2; ++v) nres[v] = addp[j + 1] ? ld_stream32(addp[j + 1] + v * 16) : zero32;
    }
#pragma unroll
    for (int c0 = 0; c0 < BN; c0 += 32) {
      uint32_t r[32];
      tmem_ld32(trow + j * BN + c0, r);
      tmem_ld_wait();
      uint4 o[4];
      if (validj[j] || STATS) {
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          float f[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) f[i] = __uint_as_float(r[g * 8 + i]);
          if (p.add_mode != 0) {
            float a[8];
            const U32B& rv = res[(c0 / 8 + g) / 2];
            unpack8((g & 1) == 0 ? rv.lo : rv.hi, a);
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] += a[i];
          }
          if (p.bias != nullptr) {  // eval mode: folded BatchNorm shift (same 8 floats for every lane: L1 broadcast)
            const float4 b0 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0 + g * 8));
            const float4 b1 = __ldg(reinterpret_cast<const float4*>(p.bias + n0 + c0 + g * 8 + 4));
            f[0] += b0.x; f[1] += b0.y; f[2] += b0.z; f[3] += b0.w;
            f[4] += b1.x; f[5] += b1.y; f[6] += b1.z; f[7] += b1.w;
          }
          if (p.relu) {
#pragma unroll
            for (int i = 0; i < 8; ++i) f[i] = fmaxf(f[i], 0.f);
          }
          o[g] = pack8(f);
        }
      }
      if (validj[j]) {  // 16 channels = one 32-byte store (a full sector per lane)
        st_global32(outp[j] + c0, o[0], o[1]);
        st_global32(outp[j] + c0 + 16, o[2], o[3]);
      }
      if (STATS && do_stats) {
        if (!validj[j]) o[0] = o[1] = o[2] = o[3] = make_uint4(0, 0, 0, 0);
        stat_chunk(scratch, lane, o, sa.s[c0 / 32], sa.q[c0 / 32]);
      }
    }
    if (p.add_mode != 0 && j + 1 < MT) {
#pragma unroll
      for (int v = 0; v < NV / 2; ++v) res[v] = nres[v];
    }
  }
}

// Window loader: padded rows [rho, rho + nrows) of the flat grid, row (n, h) at sdst + i * row_bytes.  The producer is
// ONE thread and pays ~100 clocks per TMA operation, so one-row boxes (1 KB at 7x7) made it the bottleneck wherever a
// window is many short rows — 7x7 / 9x6 maps, and every stride-2 convolution (four plane windows per slab: measured
// 32 clocks of MMA per TMA operation there, 27-40 % of the stride-1 rate).  Rows are therefore fetched as whole padded
// images (box {64, P, Hs+1, 1}: 7x7 .. 17x12 maps) or four-row bands wherever they fit inside one image, single rows
// otherwise; (n, h) advance incrementally — no division per row.  Rows h == Hs, images n < 0 or n >= N are TMA
// out-of-bounds zero fill exactly as with one-row boxes.
template <bool PAIR>
__device__ __forceinline__ void flat_load_rows(const FlatParams& p, int plane, uint32_t sdst, uint64_t* bar,
                                               uint32_t bar_cluster, int c0, int n, int h, int nrows,
                                               uint32_t row_bytes) {
  const int rows_img = p.Hs + 1;
  auto issue = [&](const CUtensorMap* m) {
    if (PAIR)
      tma2_load_4d(sdst, m, bar_cluster, c0, 0, h, n);
    else
      tma_load_4d(sdst, m, bar, c0, 0, h, n);
  };
  while (nrows > 0) {
    int took;
    if (p.use_img && h == 0 && nrows >= rows_img) {
      issue(&p.tm_ximg[plane]);
      took = rows_img;
    } else if (p.use_r4 && nrows >= 4 && h + 4 <= rows_img) {
      issue(&p.tm_x4[plane]);
      took = 4;
    } else {
      issue(&p.tm_x[plane]);
      took = 1;
    }
    sdst += took * row_bytes;
    nrows -= took;
    h += took;
    if (h >= rows_img) {
      h = 0;
      ++n;
    }
  }
}

// RES: the whole packed weight matrix of the layer (taps x slabs tiles of BN x 64) is loaded ONCE per CTA and stays in
// shared memory (64 -> 64 channel 3x3 layers: 9 tiles = 72 KB), instead of being streamed from L2 for every 256-pixel
// item: the weight ring is 2/3 of the L2 -> SM traffic of those layers.  One class, one channel tile.
// (A cluster-of-2 variant that TMA-MULTICAST each weight tile into both CTAs was validated and measured in round 2:
// 0.97-1.01x on every layer — L2 already de-duplicates concurrent requests for the same lines and every SM still
// receives and reads the whole tile — and was removed; the CTA-pair kernel below splits the tile instead.)
template <int BN, int MT, int WST, bool STATS, bool RES = false>
__global__ void __launch_bounds__(kFlatThreads, 1) conv_flat_kernel(const __grid_constant__ FlatParams p) {
  constexpr int W_BYTES = BN * 128;
  constexpr int TM = MT * 128;
  constexpr int kMaxWin = 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int w_off = p.win_stages * p.win_stage_bytes;
  const int bar_off = w_off + (RES ? p.res_tiles : WST) * W_BYTES;
  uint64_t* win_full = reinterpret_cast<uint64_t*>(smem + bar_off);
  uint64_t* win_empty = win_full + kMaxWin;
  uint64_t* w_full = win_empty + kMaxWin;
  uint64_t* w_empty = w_full + WST;
  uint64_t* tmem_full = w_empty + WST;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int tid = threadIdx.x;
  const int warp = warp_uniform_idx();
  const int slabs = p.Cs >> 6;
  const int WS = p.win_stages;
  const int item_first = int(blockIdx.x);
  const int item_stride = int(gridDim.x);
  const int mt_count = p.mtiles;  // pixel-tile slots per (class, channel tile)
  const int mt_max = p.mtiles;
  const int per_class = p.ntiles * mt_count;
  const int items_total = p.nclass * per_class;

  if (tid == 0) {
    for (int i = 0; i < kMaxWin; ++i) {
      mbar_init(&win_full[i], 1);
      mbar_init(&win_empty[i], 1);
    }
    for (int i = 0; i < WST; ++i) {
      mbar_init(&w_full[i], 1);
      mbar_init(&w_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 128);
    }
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc(tmem_slot, 2 * MT * BN);
    tmem_relinquish();
  }
  if (tid == 5 * 32) {
    tma_prefetch_desc(&p.tm_x[0]);
    tma_prefetch_desc(&p.tm_w);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);

  if (warp == 5 && elect_one()) {
    // ------------------------------ TMA producer ------------------------------
    const int rows_img = p.Hs + 1;
    const uint32_t row_bytes = (uint32_t)p.P * 128u;
    int wincount = 0, wcount = 0;
    if (RES) {  // tile (slab, tap) at index slab * ntaps + tap; one barrier for all of them
      mbar_arrive_expect_tx(&w_full[0], (uint32_t)p.res_tiles * W_BYTES);
      for (int slab = 0; slab < slabs; ++slab)
        for (int t = 0; t < p.ntaps[0]; ++t)
          tma_load_2d(smem_base + w_off + (slab * p.ntaps[0] + t) * W_BYTES, &p.tm_w, &w_full[0],
                      p.taps[0][t].wk + slab * 64, 0);
    }
    for (int item = item_first; item < items_total; item += item_stride) {
      const int cls = item / per_class;
      const int rem = item - cls * per_class;
      const int nt = rem / mt_count;
      const int mt_i = rem - nt * mt_count;
      const int q0 = (p.rev ? mt_max - 1 - mt_i : mt_i) * TM;
      const int n0 = nt * BN;
      const int rho_a = floor_div(q0 + p.smin, p.P);
      const int rho_b = floor_div(q0 + TM + p.smax - 1, p.P);
      const int nrows = rho_b - rho_a + 1;
      const int n_a = floor_div(rho_a, rows_img), h_a = rho_a - n_a * rows_img;
      const int ngrp = p.ngroups[cls];
      for (int slab = 0; slab < slabs; ++slab) {
        for (int g = 0; g < ngrp; ++g, ++wincount) {
          const int ws = wincount % WS;
          if (wincount >= WS) mbar_wait(&win_empty[ws], ((wincount / WS) - 1) & 1);
          mbar_arrive_expect_tx(&win_full[ws], (uint32_t)nrows * row_bytes);
          flat_load_rows<false>(p, p.gplane[cls][g], smem_base + ws * p.win_stage_bytes, &win_full[ws], 0u, slab * 64,
                                n_a, h_a, nrows, row_bytes);
          if (!RES)
            for (int t = p.gtap0[cls][g]; t < p.gtap0[cls][g + 1]; ++t, ++wcount) {
              const int st = wcount % WST;
              if (wcount >= WST) mbar_wait(&w_empty[st], ((wcount / WST) - 1) & 1);
              mbar_arrive_expect_tx(&w_full[st], W_BYTES);
              tma_load_2d(smem_base + w_off + st * W_BYTES, &p.tm_w, &w_full[st], p.taps[cls][t].wk + slab * 64, n0);
            }
        }
      }
    }
  } else if (warp == 4 && elect_one()) {
    // ------------------------------ MMA issuer ------------------------------
    // The single issuing thread is instruction-latency bound (an N=64 MMA retires in 32 clocks), so every
    // operand must live in uniform registers.  The TMEM base read from shared memory would not (ptxas emits
    // an ELECT/R2UR waterfall per MMA), but the kernel is the only TMEM user of its SM (kFlatSmemFloor, enforced at
    // launch: see launch_flat), so the allocation always starts at column 0: check it once and use the constant.
    if (tmem_base != 0) {
      printf("gdl: conv_flat expects TMEM base 0, got %u\n", tmem_base);
      __trap();
    }
    constexpr uint32_t idesc = make_idesc_bf16(128, BN, 0, 0);
    const uint32_t ab_hi = desc_hi_sw128(1024);
    const uint32_t a_lo0 = desc_lo_sw128(smem_base, 16), b_lo0 = desc_lo_sw128(smem_base + w_off, 16);
    int wincount = 0, wcount = 0, it = 0;
    if (RES) {
      mbar_wait(&w_full[0], 0);
      tc_fence_after();
    }
    for (int item = item_first; item < items_total; item += item_stride, ++it) {
      const int cls = item / per_class;
      const int rem = item - cls * per_class;
      const int nt = rem / mt_count;
      const int mt_i = rem - nt * mt_count;
      const int q0 = (p.rev ? mt_max - 1 - mt_i : mt_i) * TM;
      const int rho_a = floor_div(q0 + p.smin, p.P);
      const int o = q0 + p.smin - rho_a * p.P;  // first window row inside the stage
      const int acc = it & 1;
      if (it >= 2) {
        mbar_wait(&tmem_empty[acc], ((it >> 1) - 1) & 1);
        tc_fence_after();
      }
      const uint32_t d_tmem = acc * (MT * BN);
      const int ngrp = p.ngroups[cls];
      for (int slab = 0; slab < slabs; ++slab) {
        for (int g = 0; g < ngrp; ++g, ++wincount) {
          const int ws = wincount % WS;
          mbar_wait(&win_full[ws], (wincount / WS) & 1);
          tc_fence_after();
          const uint32_t a_win = a_lo0 + ((ws * p.win_stage_bytes) >> 4) + (o - p.smin) * 8;
          for (int t = p.gtap0[cls][g]; t < p.gtap0[cls][g + 1]; ++t, ++wcount) {
            const int st = RES ? slab * p.ntaps[0] + t : wcount % WST;
            if (!RES) {
              mbar_wait(&w_full[st], (wcount / WST) & 1);
              tc_fence_after();
            }
            const uint32_t a_lo = a_win + p.taps[cls][t].shift * 8;
            const uint32_t b_lo = b_lo0 + st * (W_BYTES >> 4);
            const uint32_t first = (slab | t) != 0 ? 1u : 0u;
#pragma unroll
            for (int j = 0; j < MT; ++j) {
              mma_bf16_ss(d_tmem + j * BN, desc_join(a_lo + j * 1024, ab_hi), desc_join(b_lo, ab_hi), idesc, first);
#pragma unroll
              for (int k = 1; k < 4; ++k)
                mma_bf16_acc(d_tmem + j * BN, desc_join(a_lo + j * 1024 + 2 * k, ab_hi),
                             desc_join(b_lo + 2 * k, ab_hi), idesc);
            }
            if (!RES) mma_commit(&w_empty[st]);
          }
          mma_commit(&win_empty[ws]);
        }
      }
      mma_commit(&tmem_full[acc]);
    }
  } else if (warp < 4) {
    // ------------------------------ epilogue ------------------------------
    const int lane = tid & 31;
    StatAcc<BN> sa;
#pragma unroll
    for (int c = 0; c < BN / 32; ++c) sa.s[c][0] = sa.s[c][1] = sa.q[c][0] = sa.q[c][1] = 0.f;
    sa.nt = -1;
    // one partial row [2][Cd] per epilogue warp of every CTA
    float* st_slot = (STATS && p.stats) ? p.stats + (size_t)(blockIdx.x * 4 + warp) * 2 * p.Cd : nullptr;
    if (st_slot != nullptr)
      for (int c = lane; c < 2 * p.Cd; c += 32) st_slot[c] = 0.f;
    const uint32_t scratch = smem_base + bar_off + 512 + warp * kStatWarpBytes;
    int it = 0;
    for (int item = item_first; item < items_total; item += item_stride, ++it) {
      const int cls = item / per_class;
      const int rem = item - cls * per_class;
      const int nt = rem / mt_count;
      const int mt_i = rem - nt * mt_count;
      const int q0 = (p.rev ? mt_max - 1 - mt_i : mt_i) * TM;
      const int acc = it & 1;
      if (STATS && nt != sa.nt) {
        stat_flush<BN>(sa, st_slot, p.Cd, lane);
        sa.nt = nt;
      }
      const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16) + acc * (MT * BN);
      flat_epilogue_item<BN, MT, STATS>(p, cls, nt * BN, q0, tid, lane, &tmem_full[acc], (it >> 1) & 1, trow, scratch,
                                        st_slot != nullptr, sa);
      tc_fence_before();
      mbar_arrive(&tmem_empty[acc]);
    }
    if (STATS) stat_flush<BN>(sa, st_slot, p.Cd, lane);
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 4) tmem_dealloc(tmem_base, 2 * MT * BN);
}


// ------------------------------------------------------------------------------------------
// CTA-pair variant: tcgen05.mma.cta_group::2 (tc05.cuh).  A cluster of two CTAs (one TPC) owns 2*MT*128 CONSECUTIVE
// flat pixels of one channel tile: CTA r holds the window of its own MT*128 pixels and HALF (BN/2 rows) of every
// weight tile; the leader (rank 0) issues one M = 256 MMA per K step that reads A and its half of B from each
// CTA's shared memory and accumulates each CTA's 128 rows in that CTA's TMEM.  Per SM this halves both the weight
// bytes fetched from L2 and the B bytes read from shared memory per MMA — the two resources that hold the
// single-CTA kernel at ~55 % tensor-pipe activity (an M128 x N128 x K16 MMA reads 8 KB of operands in 64 clocks =
// the whole 128 B/clk of shared-memory bandwidth, while TMA writes the next tiles into the same memory).
// The A descriptor is shared by both CTAs, so both place the first pixel of their window at the SAME shared-memory
// offset: window rows land (P-1-o) pixel rows into the stage (o = the tile's phase inside its first padded row).
//   full barriers  (window / weights): in the LEADER, 2 arrivals (each producer announces its own bytes;
//                  both CTAs' TMA loads complete_tx on the leader's barrier: cp.async.bulk.tensor.cta_group::2)
//   empty barriers (window / weights / accumulator-ready): one per CTA, released by tcgen05.commit.cta_group::2
//                  multicast to both
//   tmem_empty     : in the leader, 8 arrivals (one per epilogue warp of both CTAs, remote arrive from the peer)
//   RES: as in the single-CTA kernel, the layer's whole packed weight matrix stays in shared memory — each CTA of the
//   pair keeps ITS HALF of every tile (64 -> 64 channel 3x3 layers: 9 x 4 KB) — so the N = 64 layers get both remedies
//   for their shared-memory-bandwidth bound: no weight ring traffic and 5 KB instead of 6 KB of operands per MMA.
template <int BN, int MT, int WST, bool STATS, bool RES = false>
__global__ void __launch_bounds__(kFlatThreads, 1) conv_flat2_kernel(const __grid_constant__ FlatParams p) {
  constexpr int HB = BN / 2;
  constexpr int W_BYTES = HB * 128;
  constexpr int TM = MT * 128;
  constexpr int kMaxWin = 4;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int w_off = p.win_stages * p.win_stage_bytes;
  const int bar_off = w_off + (RES ? p.res_tiles : WST) * W_BYTES;
  uint64_t* win_full = reinterpret_cast<uint64_t*>(smem + bar_off);
  uint64_t* win_empty = win_full + kMaxWin;
  uint64_t* w_full = win_empty + kMaxWin;
  uint64_t* w_empty = w_full + WST;
  uint64_t* tmem_full = w_empty + WST;
  uint64_t* tmem_empty = tmem_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int tid = threadIdx.x;
  const int warp = warp_uniform_idx();
  const int slabs = p.Cs >> 6;
  const int WS = p.win_stages;
  const int rank = (int)cluster_ctarank();
  const int item_first = int(blockIdx.x >> 1);
  const int item_stride = int(gridDim.x >> 1);
  const int mt_count = (p.mtiles + 1) / 2;  // pairs of pixel tiles per (class, channel tile); an odd tail tile is padding
  const int per_class = p.ntiles * mt_count;
  const int items_total = p.nclass * per_class;

  if (tid == 0) {
    for (int i = 0; i < kMaxWin; ++i) {
      mbar_init(&win_full[i], 2);
      mbar_init(&win_empty[i], 1);
    }
    for (int i = 0; i < WST; ++i) {
      mbar_init(&w_full[i], 2);
      mbar_init(&w_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&tmem_full[i], 1);
      mbar_init(&tmem_empty[i], 8);
    }
    fence_mbar_init();
  }
  if (warp == 4) {
    tmem_alloc2(tmem_slot, 2 * MT * BN);
    tmem_relinquish2();
  }
  if (tid == 5 * 32) {
    tma_prefetch_desc(&p.tm_x[0]);
    tma_prefetch_desc(&p.tm_w_half);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers exist before any remote arrive / multicast commit / remote complete_tx
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t smem_base = smem_u32(smem);

  auto tile_of = [&](int item, int& cls, int& nt, int& q0) {
    cls = item / per_class;
    const int rem = item - cls * per_class;
    nt = rem / mt_count;
    const int pr = rem - nt * mt_count;
    q0 = ((p.rev ? mt_count - 1 - pr : pr) * 2 + rank) * TM;
  };

  if (warp == 5 && elect_one()) {
    // ------------------------------ TMA producer (both CTAs) ------------------------------
    const int rows_img = p.Hs + 1;
    const uint32_t row_bytes = (uint32_t)p.P * 128u;
    int wincount = 0, wcount = 0;
    if (RES) {  // this CTA's half of tile (slab, tap) at index slab * ntaps + tap; one barrier (in the leader) for all
      const uint32_t wfull = mapa_u32(smem_u32(&w_full[0]), 0);
      mbar_arrive_expect_tx_cluster(wfull, (uint32_t)p.res_tiles * W_BYTES);
      for (int slab = 0; slab < slabs; ++slab)
        for (int t = 0; t < p.ntaps[0]; ++t)
          tma2_load_2d(smem_base + w_off + (slab * p.ntaps[0] + t) * W_BYTES, &p.tm_w_half, wfull,
                       p.taps[0][t].wk + slab * 64, rank * HB);
    }
    for (int item = item_first; item < items_total; item += item_stride) {
      int cls, nt, q0;
      tile_of(item, cls, nt, q0);
      const int n0 = nt * BN + rank * HB;
      const int rho_a = floor_div(q0 + p.smin, p.P);
      const int rho_b = floor_div(q0 + TM + p.smax - 1, p.P);
      const int nrows = rho_b - rho_a + 1;
      const int o = q0 + p.smin - rho_a * p.P;  // phase of the window's first pixel inside its first padded row
      const int n_a = floor_div(rho_a, rows_img), h_a = rho_a - n_a * rows_img;
      const int ngrp = p.ngroups[cls];
      for (int slab = 0; slab < slabs; ++slab) {
        for (int g = 0; g < ngrp; ++g, ++wincount) {
          const int ws = wincount % WS;
          if (wincount >= WS) mbar_wait(&win_empty[ws], ((wincount / WS) - 1) & 1);
          const uint32_t full = mapa_u32(smem_u32(&win_full[ws]), 0);
          mbar_arrive_expect_tx_cluster(full, (uint32_t)nrows * row_bytes);
          const uint32_t sdst = smem_base + ws * p.win_stage_bytes + (uint32_t)(p.P - 1 - o) * 128u;
          flat_load_rows<true>(p, p.gplane[cls][g], sdst, nullptr, full, slab * 64, n_a, h_a, nrows, row_bytes);
          if (!RES)
          for (int t = p.gtap0[cls][g]; t < p.gtap0[cls][g + 1]; ++t, ++wcount) {
            const int st = wcount % WST;
            if (wcount >= WST) mbar_wait(&w_empty[st], ((wcount / WST) - 1) & 1);
            const uint32_t wfull = mapa_u32(smem_u32(&w_full[st]), 0);
            mbar_arrive_expect_tx_cluster(wfull, W_BYTES);
            tma2_load_2d(smem_base + w_off + st * W_BYTES, &p.tm_w_half, wfull, p.taps[cls][t].wk + slab * 64, n0);
          }
        }
      }
    }
  } else if (warp == 4 && rank == 0 && elect_one()) {
    // ------------------------------ MMA issuer (leader only) ------------------------------
    if (tmem_base != 0) {
      printf("gdl: conv_flat2 expects TMEM base 0, got %u\n", tmem_base);
      __trap();
    }
    constexpr uint32_t idesc = make_idesc_bf16(256, BN, 0, 0);
    const uint32_t ab_hi = desc_hi_sw128(1024);
    const uint32_t a_lo0 = desc_lo_sw128(smem_base, 16), b_lo0 = desc_lo_sw128(smem_base + w_off, 16);
    int wincount = 0, wcount = 0, it = 0;
    if (RES) {
      mbar_wait(&w_full[0], 0);
      tc_fence_after();
    }
    for (int item = item_first; item < items_total; item += item_stride, ++it) {
      const int cls = item / per_class;
      const int acc = it & 1;
      if (it >= 2) {
        mbar_wait(&tmem_empty[acc], ((it >> 1) - 1) & 1);
        tc_fence_after();
      }
      const uint32_t d_tmem = acc * (MT * BN);
      const int ngrp = p.ngroups[cls];
      for (int slab = 0; slab < slabs; ++slab) {
        for (int g = 0; g < ngrp; ++g, ++wincount) {
          const int ws = wincount % WS;
          mbar_wait(&win_full[ws], (wincount / WS) & 1);
          tc_fence_after();
          // pixel q0 + shift sits (P - 1 + shift - smin) pixel rows into the stage, in both CTAs
          const uint32_t a_win = a_lo0 + ((ws * p.win_stage_bytes) >> 4) + (p.P - 1 - p.smin) * 8;
          for (int t = p.gtap0[cls][g]; t < p.gtap0[cls][g + 1]; ++t, ++wcount) {
            const int st = RES ? slab * p.ntaps[0] + t : wcount % WST;
            if (!RES) {
              mbar_wait(&w_full[st], (wcount / WST) & 1);
              tc_fence_after();
            }
            const uint32_t a_lo = a_win + p.taps[cls][t].shift * 8;
            const uint32_t b_lo = b_lo0 + st * (W_BYTES >> 4);
            const uint32_t first = (slab | t) != 0 ? 1u : 0u;
#pragma unroll
            for (int j = 0; j < MT; ++j) {
              mma2_bf16_ss(d_tmem + j * BN, desc_join(a_lo + j * 1024, ab_hi), desc_join(b_lo, ab_hi), idesc, first);
#pragma unroll
              for (int k = 1; k < 4; ++k)
                mma2_bf16_acc(d_tmem + j * BN, desc_join(a_lo + j * 1024 + 2 * k, ab_hi),
                              desc_join(b_lo + 2 * k, ab_hi), idesc);
            }
            if (!RES) mma2_commit_both(&w_empty[st]);
          }
          mma2_commit_both(&win_empty[ws]);
        }
      }
      mma2_commit_both(&tmem_full[acc]);
    }
  } else if (warp < 4) {
    // ------------------------------ epilogue (both CTAs: own 128 rows x MT) ------------------------------
    const int lane = tid & 31;
    const uint32_t empty0 = mapa_u32(smem_u32(&tmem_empty[0]), 0), empty1 = mapa_u32(smem_u32(&tmem_empty[1]), 0);
    StatAcc<BN> sa;
#pragma unroll
    for (int c = 0; c < BN / 32; ++c) sa.s[c][0] = sa.s[c][1] = sa.q[c][0] = sa.q[c][1] = 0.f;
    sa.nt = -1;
    float* st_slot = (STATS && p.stats) ? p.stats + (size_t)(blockIdx.x * 4 + warp) * 2 * p.Cd : nullptr;
    if (st_slot != nullptr)
      for (int c = lane; c < 2 * p.Cd; c += 32) st_slot[c] = 0.f;
    const uint32_t scratch = smem_base + bar_off + 512 + warp * kStatWarpBytes;
    int it = 0;
    for (int item = item_first; item < items_total; item += item_stride, ++it) {
      int cls, nt, q0;
      tile_of(item, cls, nt, q0);
      const int acc = it & 1;
      if (STATS && nt != sa.nt) {
        stat_flush<BN>(sa, st_slot, p.Cd, lane);
        sa.nt = nt;
      }
      const uint32_t trow = tmem_base + (uint32_t(warp * 32) << 16) + acc * (MT * BN);
      flat_epilogue_item<BN, MT, STATS>(p, cls, nt * BN, q0, tid, lane, &tmem_full[acc], (it >> 1) & 1, trow, scratch,
                                        st_slot != nullptr, sa);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(acc ? empty1 : empty0);
    }
    if (STATS) stat_flush<BN>(sa, st_slot, p.Cd, lane);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // no CTA exits (or frees TMEM) while the leader's MMAs may still read its shared memory
  if (warp == 4) tmem_dealloc2(tmem_base, 2 * MT * BN);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
thread_local int g_flat_last_grid = 0;  // grid of the last flat launch of this thread (partial statistics rows = 4 x grid)

template <int BN, int MT, int WST, bool RES = false>
static int launch_flat(FlatParams& p, int64_t Q, cudaStream_t s) {
  constexpr int TM = MT * 128;
  const int nrows_max = (TM + p.smax - p.smin - 1 + p.P - 1) / p.P + 1;
  p.win_stage_bytes = (nrows_max * p.P * 128 + 1023) / 1024 * 1024;
  if (RES) {
    if (p.nclass != 1 || p.Cd != BN || p.ngroups[0] != 1) return 0;
    p.res_tiles = p.ntaps[0] * (p.Cs / 64);
  }
  const bool st = p.stats != nullptr;
  const int fixed = (RES ? p.res_tiles : WST) * BN * 128 + 512 + (st ? kStatScratchBytes : 0);
  int ws = (kFlatSmemBudget - fixed) / p.win_stage_bytes;
  if (ws > 4) ws = 4;
  if (ws < 2) return 0;  // window does not fit twice: not eligible
  p.win_stages = ws;
  p.mtiles = int((Q + TM - 1) / TM);
  p.ntiles = p.Cd / BN;
  p.items_total = p.nclass * p.ntiles * p.mtiles;
  int total = ws * p.win_stage_bytes + fixed + 1024;
  // TMEM base 0 (see the MMA issuer): the kernel must be the only TMEM user on its SM.  Variants that allocate all
  // 512 columns get that from tcgen05.alloc itself (it blocks until the columns are free); the others take at
  // least kFlatSmemFloor of shared memory, which leaves < 28 KB on the SM — less than any other TMEM-using kernel of
  // this library needs (stem_fwd 104 KB, stem_wgrad 95 KB, the flat / generic GEMM kernels >= 100 KB), so none can be
  // co-resident even when the audio and visual encoders run on two streams.
  if (total < kFlatSmemFloor) total = kFlatSmemFloor;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_flat_kernel<BN, MT, WST, false, RES>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_flat_kernel<BN, MT, WST, true, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               227 * 1024);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(conv_flat)");
    attr_set = true;
  }
  int grid = p.items_total < kNumSMs ? p.items_total : kNumSMs;
  g_flat_last_grid = grid;
  if (st)
    conv_flat_kernel<BN, MT, WST, true, RES><<<grid, kFlatThreads, total, s>>>(p);
  else
    conv_flat_kernel<BN, MT, WST, false, RES><<<grid, kFlatThreads, total, s>>>(p);
  GDL_CHECK_LAUNCH("conv_flat_kernel");
  return 1;
}

// CTA-pair kernel: p.tm_w_half must hold the {64, BN/2} weight map.  Returns 0 when not eligible.
template <int BN, int MT, int WST, bool RES = false>
static int launch_flat2(FlatParams& p, int64_t Q, cudaStream_t s) {
  constexpr int TM = MT * 128;
  if (RES) {
    if (p.nclass != 1 || p.Cd != BN || p.ngroups[0] != 1) return 0;
    p.res_tiles = p.ntaps[0] * (p.Cs / 64);
  }
  const int nrows_max = (TM + p.smax - p.smin - 1 + p.P - 1) / p.P + 1;
  // + P-1 pixel rows: both CTAs of a pair start their window at the same offset whatever its phase in the padded row
  p.win_stage_bytes = ((nrows_max * p.P + p.P - 1) * 128 + 1023) / 1024 * 1024;
  const bool st = p.stats != nullptr;
  const int fixed = (RES ? p.res_tiles : WST) * (BN / 2) * 128 + 512 + (st ? kStatScratchBytes : 0);
  int ws = (kFlatSmemBudget - fixed) / p.win_stage_bytes;
  if (ws > 4) ws = 4;
  if (ws < 2) return 0;
  p.win_stages = ws;
  p.mtiles = int((Q + TM - 1) / TM);
  p.ntiles = p.Cd / BN;
  p.items_total = p.nclass * p.ntiles * p.mtiles;
  int total = ws * p.win_stage_bytes + fixed + 1024;
  if (total < kFlatSmemFloor) total = kFlatSmemFloor;  // sole TMEM user of its SM (see launch_flat)
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_flat2_kernel<BN, MT, WST, false, RES>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess)
      e = cudaFuncSetAttribute(conv_flat2_kernel<BN, MT, WST, true, RES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                               227 * 1024);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(conv_flat2)");
    attr_set = true;
  }
  const int64_t pairs = (int64_t)p.nclass * p.ntiles * ((p.mtiles + 1) / 2);
  const int grid2 = int(2 * pairs < kNumSMs ? 2 * pairs : kNumSMs) & ~1;
  if (grid2 < 2) return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid2);
  cfg.blockDim = dim3(kFlatThreads);
  cfg.dynamicSmemBytes = total;
  cfg.stream = s;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2;
  at[0].val.clusterDim.y = 1;
  at[0].val.clusterDim.z = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  g_flat_last_grid = grid2;
  cudaError_t e = st ? cudaLaunchKernelEx(&cfg, conv_flat2_kernel<BN, MT, WST, true, RES>, p)
                     : cudaLaunchKernelEx(&cfg, conv_flat2_kernel<BN, MT, WST, false, RES>, p);
  if (e != cudaSuccess) return cuda_fail(e, "conv_flat2_kernel");
  return 1;
}

thread_local int g_fused_stats_min_k = -1;  // per calling thread, like gdl_set_sweep; -1: the default (0)

// kind: 0 forward 3x3/s1, 1 dgrad 3x3/s1, 2 dgrad 3x3/s2 (parity classes), 3 single tap (1x1),
// 4 forward 3x3/s2: (Hs,Ws) is the OUTPUT grid, src is the whole input [N,Hi,Wi,Cs] (sH = Wi*Cs, sN = Hi*Wi*Cs)
// read through its four parity planes x[:, a::2, b::2, :]; tap (r,s) lives in plane ((r+1)&1, (s+1)&1).
// src is the tensor the taps slide over, viewed as [N,Hs,Ws,Cs] with element strides (sW,sH,sN);
// wt is [Cd rows][K] bf16 with k = tap*Cs + c.  Returns 1 when launched, 0 when not eligible, <0 on error.
int try_conv_flat(int kind, int N, int Hs, int Ws, int Cs, int64_t sW, int64_t sH, int64_t sN, const void* src,
                  const void* wt, int64_t wt_rows, int64_t wt_k, void* dst, int Hd, int Wd, int Cd,
                  const void* add_src, int add_mode, cudaStream_t s, float* stats, int* stats_rows, const float* bias,
                  int relu) {
  if (Cs % 64 != 0 || Cd % 64 != 0) return 0;
  const int P = Ws + 1;
  if (P > 256) return 0;
  const int64_t IS = (int64_t)(Hs + 1) * P;
  const int64_t Q = (int64_t)N * IS;
  if (Q + 2 * P + 1024 >= ((int64_t)1 << 31)) return 0;
  FlatParams p;
  memset(&p, 0, sizeof(p));
  p.dst = (bf16*)dst;
  p.add_src = (const bf16*)add_src;
  p.add_mode = add_mode;
  p.bias = bias;
  p.relu = relu;
  p.rev = g_sweep_rev;
  // BatchNorm statistics in the epilogue (stat_chunk above) for convolutions with K >= the threshold: default every
  // convolution this kernel runs (gdl_set_fused_stats_min_k(K) raises it; tests/ cover both paths).
  if (stats != nullptr && wt_k < g_fused_stats_min_k) stats = nullptr;
  p.stats = stats;
  p.N = N; p.Hs = Hs; p.Ws = Ws; p.Cs = Cs;
  p.Hd = Hd; p.Wd = Wd; p.Cd = Cd;
  p.P = P; p.IS = (int)IS;
  p.dscale = 1;
  p.nclass = 1;
  if (kind == 0 || kind == 1) {
    p.ntaps[0] = 9;
    for (int r = 0; r < 3; ++r)
      for (int c = 0; c < 3; ++c) {
        FlatTap& t = p.taps[0][r * 3 + c];
        t.shift = kind == 0 ? (r - 1) * P + (c - 1) : (1 - r) * P + (1 - c);
        t.wk = (r * 3 + c) * Cs;
      }
  } else if (kind == 2) {
    p.dscale = 2;
    p.nclass = 4;
    // order the classes heavy-first so the persistent loop's tail is made of cheap items
    const int cph[4] = {1, 1, 0, 0}, cpw[4] = {1, 0, 1, 0};
    for (int c = 0; c < 4; ++c) {
      p.ph[c] = cph[c];
      p.pw[c] = cpw[c];
      int nr = 0, rr[2], dh[2];
      if (cph[c] == 0) { rr[0] = 1; dh[0] = 0; nr = 1; } else { rr[0] = 0; dh[0] = 1; rr[1] = 2; dh[1] = 0; nr = 2; }
      int nc = 0, cc[2], dw[2];
      if (cpw[c] == 0) { cc[0] = 1; dw[0] = 0; nc = 1; } else { cc[0] = 0; dw[0] = 1; cc[1] = 2; dw[1] = 0; nc = 2; }
      int k = 0;
      for (int a = 0; a < nr; ++a)
        for (int b = 0; b < nc; ++b) {
          p.taps[c][k].shift = dh[a] * P + dw[b];
          p.taps[c][k].wk = (rr[a] * 3 + cc[b]) * Cs;
          ++k;
        }
      p.ntaps[c] = k;
    }
  } else if (kind == 4) {
    // taps grouped by plane, heavy groups first: (1,1) 4 taps, (1,0) 2, (0,1) 2, (0,0) 1
    const int pa[4] = {1, 1, 0, 0}, pb[4] = {1, 0, 1, 0};
    int k = 0;
    p.ngroups[0] = 4;
    for (int g = 0; g < 4; ++g) {
      p.gplane[0][g] = pa[g] * 2 + pb[g];
      p.gtap0[0][g] = k;
      for (int r = 0; r < 3; ++r)
        for (int c = 0; c < 3; ++c) {
          if (((r + 1) & 1) != pa[g] || ((c + 1) & 1) != pb[g]) continue;
          p.taps[0][k].shift = (r == 0 ? -1 : 0) * P + (c == 0 ? -1 : 0);
          p.taps[0][k].wk = (r * 3 + c) * Cs;
          ++k;
        }
    }
    p.gtap0[0][4] = k;
    p.ntaps[0] = k;
  } else {
    p.ntaps[0] = 1;
    p.taps[0][0].shift = 0;
    p.taps[0][0].wk = 0;
  }
  if (kind != 4)
    for (int c = 0; c < p.nclass; ++c) {
      p.ngroups[c] = 1;
      p.gplane[c][0] = 0;
      p.gtap0[c][0] = 0;
      p.gtap0[c][1] = p.ntaps[c];
    }
  p.smin = 0;
  p.smax = 0;
  for (int c = 0; c < p.nclass; ++c)
    for (int t = 0; t < p.ntaps[c]; ++t) {
      if (p.taps[c][t].shift < p.smin) p.smin = p.taps[c][t].shift;
      if (p.taps[c][t].shift > p.smax) p.smax = p.taps[c][t].shift;
    }
  const int BN = (Cd % 128 == 0) ? 128 : 64;
  // four-row boxes, and whole-image boxes for maps of at most 32 KB per slab (flat_load_rows)
  const int rows_img = Hs + 1;
  p.use_r4 = rows_img >= 4;
  p.use_img = rows_img <= 256 && (int64_t)rows_img * P * 128 <= 32 * 1024;
  auto views = [&](const void* base, int w, int h, int64_t vW, int64_t vH, int idx) -> bool {
    const CUtensorMap* t = tmap_view4(base, Cs, w, h, N, vW, vH, sN, P);
    if (!t) return false;
    p.tm_x[idx] = *t;
    if (p.use_r4) {
      if (!(t = tmap_view4(base, Cs, w, h, N, vW, vH, sN, P, 4))) return false;
      p.tm_x4[idx] = *t;
    }
    if (p.use_img) {
      if (!(t = tmap_view4(base, Cs, w, h, N, vW, vH, sN, P, rows_img))) return false;
      p.tm_ximg[idx] = *t;
    }
    return true;
  };
  if (kind == 4) {
    const int Wi = int(sH / Cs), Hi = int(sN / sH);
    for (int a = 0; a < 2; ++a)
      for (int b = 0; b < 2; ++b) {
        const int ph = (Hi - a + 1) / 2, pw = (Wi - b + 1) / 2;
        if (ph <= 0 || pw <= 0) return 0;
        if (!views((const bf16*)src + ((int64_t)a * Wi + b) * Cs, pw, ph, 2 * (int64_t)Cs, 2 * sH, a * 2 + b)) return GDL_ECUDA;
      }
  } else {
    if (!views(src, Ws, Hs, sW, sH, 0)) return GDL_ECUDA;
  }
  const CUtensorMap* tw = tmap_rows(wt, wt_rows, wt_k, BN);
  if (!tw) return GDL_ECUDA;
  p.tm_w = *tw;
  // MT = 2 halves the weight traffic per MMA (measured 1.2-1.4x on every layer of the bench geometry);
  // MT = 1 only when the problem would not fill one wave of CTAs otherwise
  // Tile shape by a wave-count model (small per-GPU batches: layer3/4 have a few hundred tiles, and a static
  // persistent grid pays whole rounds).  Relative cost of one round: a single CTA with MT = 1 pays the full weight
  // stream per 128 pixels (1.15), MT = 2 shares it (2.0 for twice the pixels), a CTA pair halves it again (1.7).
  const int64_t per_px = (int64_t)p.nclass * (Cd / BN);
  const int64_t items2 = per_px * ((Q + 255) / 256), items1 = per_px * ((Q + 127) / 128);
  const int64_t pairs2 = per_px * ((Q + 511) / 512);
  const double cost_mt2 = 2.0 * double((items2 + kNumSMs - 1) / kNumSMs);
  const double cost_mt1 = 1.15 * double((items1 + kNumSMs - 1) / kNumSMs);
  const double cost_pair = 1.7 * double((pairs2 + kNumSMs / 2 - 1) / (kNumSMs / 2));
  const int mt = cost_mt2 <= cost_mt1 ? 2 : 1;
  const bool pair_wins = cost_pair <= (mt == 2 ? cost_mt2 : cost_mt1);
  int rc = 0;
  if (pair_wins) {  // CTA-pair kernel (cta_group::2) where the wave-count model above prefers it
    const CUtensorMap* th = tmap_rows(wt, wt_rows, wt_k, BN / 2);
    if (!th) return GDL_ECUDA;
    p.tm_w_half = *th;
  }
  if (BN == 128) {
    if (pair_wins) rc = launch_flat2<128, 2, 6>(p, Q, s);
    if (rc == 0 && mt == 2) rc = launch_flat<128, 2, 4>(p, Q, s);
    if (rc == 0) rc = launch_flat<128, 1, 4>(p, Q, s);
  } else {
    // 64 -> 64 channel 3x3 layers keep their 72 KB of weights in shared memory (resident; measured: 56x56 forward /
    // dgrad 700-730 -> 800+ TF, step 23.11 -> 22.82 ms), as a CTA pair where the model prefers one.  The CTA pair
    // also serves the other 64-channel tiles (e.g. the 128 -> 64 channel stride-2 data gradients): N = 64 MMAs read
    // 6 KB of operands per 32 clocks on one SM, 5 KB as a pair.
    const bool res_ok = mt == 2 && Cs == 64 && Cd == 64 && (kind == 0 || kind == 1);
    if (pair_wins) rc = res_ok ? launch_flat2<64, 2, 8, true>(p, Q, s) : launch_flat2<64, 2, 8>(p, Q, s);
    if (rc == 0 && res_ok) rc = launch_flat<64, 2, 6, true>(p, Q, s);
    if (rc == 0 && mt == 2) rc = launch_flat<64, 2, 6>(p, Q, s);
    if (rc == 0) rc = launch_flat<64, 1, 6>(p, Q, s);
  }
  // one partial row per epilogue warp of every CTA of the grid that ran
  if (rc > 0 && stats_rows != nullptr && stats != nullptr) *stats_rows = g_flat_last_grid * 4;
  return rc;
}

}  // namespace gdl

extern "C" int gdl_set_fused_stats_min_k(int k) {
  int old = gdl::g_fused_stats_min_k;
  gdl::g_fused_stats_min_k = k < 0 ? -1 : k;
  return old;
}
