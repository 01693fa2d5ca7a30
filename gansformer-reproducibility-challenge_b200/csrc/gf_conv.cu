// gf_conv.cu -- row f1, first kernel: the 3x3 stride-1 convolution of the synthesis layers as a tcgen05 implicit GEMM (TF32),
// channels-last, no im2col buffer.
//
// Replaces, on the reference side (expected src/training/network.py, not in the checkout): the convolution inside
// modulated_conv2d_layer in its activation-scaling form -- the caller has already multiplied x by the style (the attention
// kernel's store side does that) and applies the demodulation afterwards (the attention kernel's load side) -- so the weights
// are batch-shared and the op is a plain  y[b,h,w,o] = sum_{dy,dx,i} x[b,h+dy-1,w+dx-1,i] * wt[dy*3+dx][o][i]  with zero padding.
//
// GEMM view: M = output pixels (one CTA tile = an 8 x 16 patch = 128 pixels), N = output channels (BN = 64 / 128 / 256 per tile),
// K = 9 taps x Cin.  Per K step (one tap, 32 input channels):
//   warp 0   TMA producer: the A operand is a 4-D box {32 ch, 16 w, 8 h, 1 b} of x at (h0+dy-1, w0+dx-1) -- out-of-image
//            coordinates are zero-filled by TMA, which IS the padding -- landing as 128 rows x 128 B, SWIZZLE_128B (K-major);
//            the B operand is a 2-D box {32 ch, BN rows} of the packed weights wt[tap] (K-major, SWIZZLE_128B)
//   warp 1   MMA issuer (warp-converged, uniform-register descriptors): 4 x tcgen05.mma kind::tf32 (M=128, N=BN, K=8) per step into
//            one of two TMEM accumulators (the epilogue of tile i overlaps the MMAs of tile i+1)
//   warps 2-5 epilogue: TMEM -> registers -> swizzled staging slab (128 pixels x 32 ch) -> TMA 4-D store, two slabs in flight
// Persistent grid (one CTA per SM), tiles handed out round-robin with the N tile innermost.
// Two kernels: version 1 below fetches every tap's A box separately (9 reads of each input byte from L2) and is bound by the
// L2 -> shared-memory path; version 2 further down shares one activation box per filter column among its three taps (3.4 reads) and
// is bound by the tensor pipe (ncu: 84-89 % active).  The dispatch at the bottom picks per shape from measurements: version 2 wherever
// the grid fills the GPU, version 1 for small grids (res 16) and, with 256 x 256 tiles, for Cin >= 512 (res 64).  Against cuDNN's
// TF32 kernels on the generator's five stride-1 layers (batch 32): 2.50-2.63 ms vs 2.48-2.50 ms in total (DESIGN.md 9.9).
#include <stdlib.h>
#include <string.h>
#include "gf_common.cuh"
#include "gf_tc_common.cuh"
#include "../../include/gf_ops.h"

namespace gf {
namespace cv {

using namespace tc;

constexpr int PH = 8, PW = 16, TILE_M = PH * PW;      // output patch of one tile
constexpr int BK = 32;                               // input channels per K step = one 128-byte swizzle span
constexpr int A_BYTES = TILE_M * BK * 4;             // 16 KB
constexpr int NUM_THREADS = 192;
constexpr int MAX_STAGES = 8;

struct Bars {
  uint64_t full[MAX_STAGES], empty[MAX_STAGES];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_base, pad;
};

struct Params {
  int B, H, W, Cin, Cout;
  int tiles_h, tiles_w, tiles_n;       // patches per image column / row, N tiles
  long long total_tiles;
  int nstages;
  float alpha;                         // TF32 truncation-bias compensation of the streamed operand
};

// 4-D tiled load: coordinates {c, w, h, b} (innermost first); out-of-bounds elements are zero-filled
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}

// MT = M tiles (8 x 16 patches, stacked in h) per CTA tile: with MT = 2 the two 128-pixel halves of a 16 x 16 patch share every weight
// slab (one B load, two MMAs into two accumulators) -- the flops per loaded byte go up by a third when BN is small
// NBUF = TMEM accumulator sets: 2 overlaps the epilogue of a tile with the MMAs of the next; 1 lets a tile use all 512 columns
// (256 pixels x 256 channels: a third less L2 -> shared-memory traffic per flop, epilogue exposed)
template <int BN, int MT, int NBUF>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv3x3_tc_kernel(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmY,
                  const Params P) {
  constexpr int B_BYTES = BN * BK * 4;
  constexpr int STAGE_BYTES = MT * A_BYTES + B_BYTES;
  constexpr int ACC_COLS = MT * BN;                                        // TMEM columns of one tile's accumulators
  constexpr int TMEM_COLS = NBUF * ACC_COLS <= 128 ? 128 : (NBUF * ACC_COLS <= 256 ? 256 : 512);
  static_assert(NBUF * ACC_COLS <= 512, "accumulators exceed TMEM");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t s_base = smem_u32(smem);
  const int nst = P.nstages;
  const uint32_t s_out = s_base + (uint32_t)nst * STAGE_BYTES;             // two staging slabs of 16 KB
  Bars* bars = reinterpret_cast<Bars*>(smem + (size_t)nst * STAGE_BYTES + 2 * A_BYTES);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int ksteps = 9 * (P.Cin / BK);

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmX); prefetch_tmap(&tmW); prefetch_tmap(&tmY);
    for (int i = 0; i < nst; ++i) { mbar_init(smem_u32(&bars->full[i]), 1); mbar_init(smem_u32(&bars->empty[i]), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&bars->acc_full[i]), 1); mbar_init(smem_u32(&bars->acc_empty[i]), 4); }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, bars->tmem_base, 0);

  // tile index -> (n tile, patch w, patch h, image); the N tile is innermost so neighbouring CTAs share their input patch in L2
  auto decode = [&](long long t, int& nt, int& pw, int& ph, int& b) {
    nt = (int)(t % P.tiles_n); t /= P.tiles_n;
    pw = (int)(t % P.tiles_w); t /= P.tiles_w;
    ph = (int)(t % P.tiles_h); b = (int)(t / P.tiles_h);
  };

  if (warp == 0) {
    // =============================== TMA producer ===============================
    if (lane == 0) {
      int stage = 0; uint32_t ph_ = 0;
      for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
        int nt, pw, ph, b;
        decode(t, nt, pw, ph, b);
        const int h0 = ph * PH * MT, w0 = pw * PW, n0 = nt * BN;
        for (int tap = 0; tap < 9; ++tap) {
          const int dy = tap / 3, dx = tap - dy * 3;
          for (int c0 = 0; c0 < P.Cin; c0 += BK) {
            mbar_wait(smem_u32(&bars->empty[stage]), ph_ ^ 1u);
            const uint32_t fb = smem_u32(&bars->full[stage]);
            mbar_expect_tx(fb, (uint32_t)STAGE_BYTES);
            const uint32_t sa = s_base + (uint32_t)stage * STAGE_BYTES;
            tma_load_4d(sa, &tmX, fb, c0, w0 + dx - 1, h0 + dy - 1, b);           // zero-filled outside the image = the padding
            tma_load_2d(sa + MT * A_BYTES, &tmW, fb, c0, tap * P.Cout + n0);      // (the A box is {32, 16, 8 * MT, 1}: MT stacked patches)
            if (++stage == nst) { stage = 0; ph_ ^= 1u; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (warp-converged) ===============================
    constexpr uint32_t IDESC = umma_idesc_tf32(TILE_M, BN);
    const uint64_t dA0 = umma_desc(s_base, 1024, LAYOUT_SW128);
    const uint64_t dB0 = umma_desc(s_base + MT * A_BYTES, 1024, LAYOUT_SW128);
    int stage = 0; uint32_t ph_ = 0;
    uint32_t it = 0;
    for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x, ++it) {
      const int buf = (int)(it % NBUF);
      mbar_wait(smem_u32(&bars->acc_empty[buf]), ((it / NBUF) & 1u) ^ 1u);        // epilogue of the tile NBUF iterations back is done
      tc_fence_after();
      const uint32_t d_acc = tmem + (uint32_t)buf * ACC_COLS;
#pragma unroll 1
      for (int ks = 0; ks < ksteps; ++ks) {
        mbar_wait(smem_u32(&bars->full[stage]), ph_);
        tc_fence_after();
        const uint64_t da = dA0 + (uint64_t)(stage * (STAGE_BYTES >> 4));
        const uint64_t db = dB0 + (uint64_t)(stage * (STAGE_BYTES >> 4));
#pragma unroll
        for (int mt = 0; mt < MT; ++mt)
#pragma unroll
          for (int kk = 0; kk < 4; ++kk)
            umma_ss_elect(d_acc + mt * BN, da + (uint64_t)(mt * (A_BYTES >> 4)) + kk * 2, db + kk * 2, IDESC, (ks | kk) ? 1u : 0u);
        umma_commit_elect(smem_u32(&bars->empty[stage]));
        if (++stage == nst) { stage = 0; ph_ ^= 1u; }
      }
      umma_commit_elect(smem_u32(&bars->acc_full[buf]));
    }
  } else {
    // =============================== epilogue warps ===============================
    const int q = warp & 3;                                   // TMEM lane quadrant
    const int row = q * 32 + lane;                            // pixel inside the patch: (row / 16, row % 16)
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int sw = row & 7;
    const bool leader = warp == 2 && lane == 0;
    uint32_t it = 0, slab_ctr = 0;
    for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x, ++it) {
      int nt, pw, ph, b;
      decode(t, nt, pw, ph, b);
      const int buf = (int)(it % NBUF);
      mbar_wait(smem_u32(&bars->acc_full[buf]), (it / NBUF) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < MT * BN; cc += 32, ++slab_ctr) {
        const int mt = cc / BN, c0 = cc - mt * BN;             // accumulator of patch mt, output channels c0 .. c0 + 31
        float v[32];
        tmem_ld16(tmem + lane_addr + (uint32_t)buf * ACC_COLS + cc, v);
        tmem_ld16(tmem + lane_addr + (uint32_t)buf * ACC_COLS + cc + 16, v + 16);
        tmem_wait_ld();
        const int sl = (int)(slab_ctr & 1u);
        if (slab_ctr >= 2) {                                   // the store that last read this staging slab has finished reading it
          if (leader) tma_wait_read1();
          named_bar_sync(1, 128);
        }
        uint8_t* dst = smem + (size_t)nst * STAGE_BYTES + (size_t)sl * A_BYTES + (size_t)row * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          *reinterpret_cast<float4*>(dst + ((c ^ sw) << 4)) =
              make_float4(v[c * 4] * P.alpha, v[c * 4 + 1] * P.alpha, v[c * 4 + 2] * P.alpha, v[c * 4 + 3] * P.alpha);
        fence_proxy_async();
        named_bar_sync(2, 128);
        if (leader) {
          tma_store_4d(&tmY, s_out + (uint32_t)sl * A_BYTES, nt * BN + c0, pw * PW, (ph * MT + mt) * PH, b);
          tma_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->acc_empty[buf]));
    }
    if (leader) tma_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS) : "memory");
  }
}

// ---------------------------------------------------------------------------------------------------------
// Version 2: the three taps of a filter COLUMN share one activation box.  For a fixed dx the boxes of dy = 0, 1, 2 are the same
// pixels shifted by whole image rows, and one image row of the 16-wide patch is 16 shared-memory rows = 2 KB -- a multiple of the
// 1 KB swizzle repeat.  So one {32 ch, 16 w, 8 MT + 2 h} box per (dx, channel slab) serves all three dy taps (and both stacked
// patches) through UMMA descriptors that differ only by (dy + 8 mt) * 2048 bytes: the activation traffic from L2 drops from 9 to
// 3 * (8 MT + 2) / (8 MT) reads per input byte (3.4 for MT = 2), which is what bounded version 1.  Weights have their own ring
// (one [BN x 32] slab per tap and channel slab).
// ---------------------------------------------------------------------------------------------------------
constexpr int MAX_STA = 4, MAX_STB = 6;
struct Bars2 {
  uint64_t fullA[MAX_STA], emptyA[MAX_STA];
  uint64_t fullB[MAX_STB], emptyB[MAX_STB];
  uint64_t acc_full[2], acc_empty[2];
  uint32_t tmem_base, pad;
};
struct Params2 {
  int B, H, W, Cin, Cout;
  int tiles_h, tiles_w, tiles_n;
  long long total_tiles;
  int nsta, nstb;
  float alpha;
};

template <int BN, int MT, int NBUF>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv3x3_tc_kernel_v2(const __grid_constant__ CUtensorMap tmX, const __grid_constant__ CUtensorMap tmW, const __grid_constant__ CUtensorMap tmY,
                     const Params2 P) {
  constexpr int A2_BYTES = (PH * MT + 2) * PW * 128;                         // halo box: (8 MT + 2) image rows x 16 pixels x 128 B
  constexpr int B_BYTES = BN * BK * 4;
  constexpr int ACC_COLS = MT * BN;
  constexpr int TMEM_COLS = NBUF * ACC_COLS <= 128 ? 128 : (NBUF * ACC_COLS <= 256 ? 256 : 512);
  static_assert(NBUF * ACC_COLS <= 512, "accumulators exceed TMEM");
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const uint32_t s_base = smem_u32(smem);
  const int nsta = P.nsta, nstb = P.nstb;
  const uint32_t s_a = s_base, s_b = s_base + (uint32_t)nsta * A2_BYTES;
  const uint32_t s_out = s_b + (uint32_t)nstb * B_BYTES;                     // two staging slabs of 16 KB
  uint8_t* out_ptr = smem + (size_t)nsta * A2_BYTES + (size_t)nstb * B_BYTES;
  Bars2* bars = reinterpret_cast<Bars2*>(out_ptr + 2 * A_BYTES);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int nslab = P.Cin / BK;

  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmX); prefetch_tmap(&tmW); prefetch_tmap(&tmY);
    for (int i = 0; i < nsta; ++i) { mbar_init(smem_u32(&bars->fullA[i]), 1); mbar_init(smem_u32(&bars->emptyA[i]), 1); }
    for (int i = 0; i < nstb; ++i) { mbar_init(smem_u32(&bars->fullB[i]), 1); mbar_init(smem_u32(&bars->emptyB[i]), 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&bars->acc_full[i]), 1); mbar_init(smem_u32(&bars->acc_empty[i]), 4); }
    fence_barrier_init();
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&bars->tmem_base)), "n"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = __shfl_sync(0xffffffffu, bars->tmem_base, 0);

  auto decode = [&](long long t, int& nt, int& pw, int& ph, int& b) {
    nt = (int)(t % P.tiles_n); t /= P.tiles_n;
    pw = (int)(t % P.tiles_w); t /= P.tiles_w;
    ph = (int)(t % P.tiles_h); b = (int)(t / P.tiles_h);
  };

  if (warp == 0) {
    // =============================== TMA producer: loads in the order the MMA warp consumes them ===============================
    if (lane == 0) {
      int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
      for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x) {
        int nt, pw, ph, b;
        decode(t, nt, pw, ph, b);
        const int h0 = ph * PH * MT, w0 = pw * PW, n0 = nt * BN;
        for (int sl = 0; sl < nslab; ++sl) {
          for (int dx = 0; dx < 3; ++dx) {
            mbar_wait(smem_u32(&bars->emptyA[sa]), pa ^ 1u);
            const uint32_t fa = smem_u32(&bars->fullA[sa]);
            mbar_expect_tx(fa, (uint32_t)A2_BYTES);
            tma_load_4d(s_a + (uint32_t)sa * A2_BYTES, &tmX, fa, sl * BK, w0 + dx - 1, h0 - 1, b);      // rows h0-1 .. h0+8MT: zero-filled outside
            if (++sa == nsta) { sa = 0; pa ^= 1u; }
            for (int dy = 0; dy < 3; ++dy) {
              mbar_wait(smem_u32(&bars->emptyB[sb]), pb ^ 1u);
              const uint32_t fb = smem_u32(&bars->fullB[sb]);
              mbar_expect_tx(fb, (uint32_t)B_BYTES);
              tma_load_2d(s_b + (uint32_t)sb * B_BYTES, &tmW, fb, sl * BK, (dy * 3 + dx) * P.Cout + n0);
              if (++sb == nstb) { sb = 0; pb ^= 1u; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // =============================== MMA issuer (warp-converged) ===============================
    constexpr uint32_t IDESC = umma_idesc_tf32(TILE_M, BN);
    const uint64_t dA0 = umma_desc(s_a, 1024, LAYOUT_SW128);
    const uint64_t dB0 = umma_desc(s_b, 1024, LAYOUT_SW128);
    int sa = 0, sb = 0; uint32_t pa = 0, pb = 0;
    uint32_t it = 0;
    for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x, ++it) {
      const int buf = (int)(it % NBUF);
      mbar_wait(smem_u32(&bars->acc_empty[buf]), ((it / NBUF) & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_acc = tmem + (uint32_t)buf * ACC_COLS;
      uint32_t first = 0;                                      // 0 until the tile's first MMA has been issued
#pragma unroll 1
      for (int sl = 0; sl < nslab; ++sl) {
#pragma unroll 1
        for (int dx = 0; dx < 3; ++dx) {
          mbar_wait(smem_u32(&bars->fullA[sa]), pa);
          tc_fence_after();
          const uint64_t da = dA0 + (uint64_t)(sa * (A2_BYTES >> 4));
#pragma unroll 1
          for (int dy = 0; dy < 3; ++dy) {
            mbar_wait(smem_u32(&bars->fullB[sb]), pb);
            tc_fence_after();
            const uint64_t db = dB0 + (uint64_t)(sb * (B_BYTES >> 4));
#pragma unroll
            for (int mt = 0; mt < MT; ++mt)
#pragma unroll
              for (int kk = 0; kk < 4; ++kk) {
                // patch mt, tap row dy: the box shifted down by (dy + 8 mt) image rows of 16 pixels x 128 B = 2 KB each
                umma_ss_elect(d_acc + mt * BN, da + (uint64_t)(((dy + PH * mt) * PW * 128) >> 4) + kk * 2, db + kk * 2, IDESC, first | (uint32_t)kk);
              }
            first = 1;
            umma_commit_elect(smem_u32(&bars->emptyB[sb]));
            if (++sb == nstb) { sb = 0; pb ^= 1u; }
          }
          umma_commit_elect(smem_u32(&bars->emptyA[sa]));
          if (++sa == nsta) { sa = 0; pa ^= 1u; }
        }
      }
      umma_commit_elect(smem_u32(&bars->acc_full[buf]));
    }
  } else {
    // =============================== epilogue warps (as version 1) ===============================
    const int q = warp & 3;
    const int row = q * 32 + lane;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    const int sw = row & 7;
    const bool leader = warp == 2 && lane == 0;
    uint32_t it = 0, slab_ctr = 0;
    for (long long t = blockIdx.x; t < P.total_tiles; t += gridDim.x, ++it) {
      int nt, pw, ph, b;
      decode(t, nt, pw, ph, b);
      const int buf = (int)(it % NBUF);
      mbar_wait(smem_u32(&bars->acc_full[buf]), (it / NBUF) & 1u);
      tc_fence_after();
#pragma unroll 1
      for (int cc = 0; cc < MT * BN; cc += 32, ++slab_ctr) {
        const int mt = cc / BN, c0 = cc - mt * BN;
        float v[32];
        tmem_ld16(tmem + lane_addr + (uint32_t)buf * ACC_COLS + cc, v);
        tmem_ld16(tmem + lane_addr + (uint32_t)buf * ACC_COLS + cc + 16, v + 16);
        tmem_wait_ld();
        const int sl = (int)(slab_ctr & 1u);
        if (slab_ctr >= 2) {
          if (leader) tma_wait_read1();
          named_bar_sync(1, 128);
        }
        uint8_t* dst = out_ptr + (size_t)sl * A_BYTES + (size_t)row * 128;
#pragma unroll
        for (int c = 0; c < 8; ++c)
          *reinterpret_cast<float4*>(dst + ((c ^ sw) << 4)) =
              make_float4(v[c * 4] * P.alpha, v[c * 4 + 1] * P.alpha, v[c * 4 + 2] * P.alpha, v[c * 4 + 3] * P.alpha);
        fence_proxy_async();
        named_bar_sync(2, 128);
        if (leader) {
          tma_store_4d(&tmY, s_out + (uint32_t)sl * A_BYTES, nt * BN + c0, pw * PW, (ph * MT + mt) * PH, b);
          tma_commit();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&bars->acc_empty[buf]));
    }
    if (leader) tma_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "n"(TMEM_COLS) : "memory");
  }
}

// 4-D fp32 NHWC tensor map: dims {C, W, H, B}, box {box_c, box_w, box_h, 1}
static int make_map_nhwc(CUtensorMap* m, const void* base, int B, int H, int W, int C, int box_c, int box_w, int box_h) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { set_error("cuTensorMapEncodeTiled entry point not available"); return GF_ERR_CUDA; }
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  cuuint64_t strides[3] = {(cuuint64_t)C * 4, (cuuint64_t)W * C * 4, (cuuint64_t)H * W * C * 4};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)box_w, (cuuint32_t)box_h, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (NHWC 4-D) failed with CUresult %d (B=%d H=%d W=%d C=%d)", (int)r, B, H, W, C); return GF_ERR_CUDA; }
  return GF_OK;
}

template <int BN, int MT, int NBUF>
static int launch(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout, cudaStream_t st) {
  constexpr int B_BYTES = BN * BK * 4, STAGE_BYTES = MT * A_BYTES + B_BYTES;
  CUtensorMap tmX, tmW, tmY;
  int rc;
  if ((rc = make_map_nhwc(&tmX, x, B, H, W, Cin, BK, PW, PH * MT))) return rc;
  if ((rc = make_map(&tmW, wt, (uint64_t)9 * Cout, (uint64_t)Cin, BN, BK, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_nhwc(&tmY, y, B, H, W, Cout, 32, PW, PH))) return rc;
  Params P;
  P.B = B; P.H = H; P.W = W; P.Cin = Cin; P.Cout = Cout;
  P.tiles_h = H / (PH * MT); P.tiles_w = W / PW; P.tiles_n = Cout / BN;
  P.total_tiles = (long long)B * P.tiles_h * P.tiles_w * P.tiles_n;
  int nst = (device_smem_optin() - 2 * A_BYTES - (int)sizeof(Bars) - 1024) / STAGE_BYTES;
  if (nst > MAX_STAGES) nst = MAX_STAGES;
  if (nst < 2) { set_error("conv3x3: shared memory too small"); return GF_ERR_UNSUPPORTED; }
  P.nstages = nst;
  P.alpha = 1.000352220f;              // the tensor core truncates x to TF32 (mean relative bias 0.7213 * 2^-11); the weights are pre-rounded
  const int smem_bytes = nst * STAGE_BYTES + 2 * A_BYTES + (int)sizeof(Bars) + 1024;
  auto kern = conv3x3_tc_kernel<BN, MT, NBUF>;
  GF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  long long grid = device_sms();
  if (grid > P.total_tiles) grid = P.total_tiles;
  kern<<<(unsigned)grid, NUM_THREADS, smem_bytes, st>>>(tmX, tmW, tmY, P);
  GF_LAUNCH_OK();
  return GF_OK;
}

template <int BN, int MT, int NBUF>
static int launch_v2(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout, cudaStream_t st) {
  constexpr int A2_BYTES = (PH * MT + 2) * PW * 128, B_BYTES = BN * BK * 4;
  CUtensorMap tmX, tmW, tmY;
  int rc;
  if ((rc = make_map_nhwc(&tmX, x, B, H, W, Cin, BK, PW, PH * MT + 2))) return rc;
  if ((rc = make_map(&tmW, wt, (uint64_t)9 * Cout, (uint64_t)Cin, BN, BK, CU_TENSOR_MAP_SWIZZLE_128B))) return rc;
  if ((rc = make_map_nhwc(&tmY, y, B, H, W, Cout, 32, PW, PH))) return rc;
  Params2 P;
  P.B = B; P.H = H; P.W = W; P.Cin = Cin; P.Cout = Cout;
  P.tiles_h = H / (PH * MT); P.tiles_w = W / PW; P.tiles_n = Cout / BN;
  P.total_tiles = (long long)B * P.tiles_h * P.tiles_w * P.tiles_n;
  // shared memory: activation ring (one box per filter column) + weight ring (three slabs per box) + two staging slabs
  const int avail = device_smem_optin() - 2 * A_BYTES - (int)sizeof(Bars2) - 1024;
  int nsta = 2, nstb = (avail - nsta * A2_BYTES) / B_BYTES;
  if (nstb > MAX_STB) {                                   // room to spare: a third activation stage
    nsta = 3;
    nstb = (avail - nsta * A2_BYTES) / B_BYTES;
    if (nstb > MAX_STB) nstb = MAX_STB;
  }
  if (nstb < 2) { set_error("conv3x3 v2: shared memory too small (BN=%d MT=%d)", BN, MT); return GF_ERR_UNSUPPORTED; }
  P.nsta = nsta; P.nstb = nstb;
  P.alpha = 1.000352220f;
  const int smem_bytes = nsta * A2_BYTES + nstb * B_BYTES + 2 * A_BYTES + (int)sizeof(Bars2) + 1024;
  auto kern = conv3x3_tc_kernel_v2<BN, MT, NBUF>;
  GF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
  long long grid = device_sms();
  if (grid > P.total_tiles) grid = P.total_tiles;
  kern<<<(unsigned)grid, NUM_THREADS, smem_bytes, st>>>(tmX, tmW, tmY, P);
  GF_LAUNCH_OK();
  return GF_OK;
}

// The twelve instantiations, addressed by (version, BN, MT); NBUF follows from them (one accumulator set only for 256 x 256 tiles)
typedef int (*LaunchFn)(const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
struct Variant { int version, bn, mt; LaunchFn fn; };
static const Variant kVariants[] = {
    {1, 256, 2, launch<256, 2, 1>},    {1, 256, 1, launch<256, 1, 2>},    {1, 128, 2, launch<128, 2, 2>},
    {1, 128, 1, launch<128, 1, 2>},    {1, 64, 2, launch<64, 2, 2>},      {1, 64, 1, launch<64, 1, 2>},
    {2, 256, 2, launch_v2<256, 2, 1>}, {2, 256, 1, launch_v2<256, 1, 2>}, {2, 128, 2, launch_v2<128, 2, 2>},
    {2, 128, 1, launch_v2<128, 1, 2>}, {2, 64, 2, launch_v2<64, 2, 2>},   {2, 64, 1, launch_v2<64, 1, 2>},
};

static const Variant* find_variant(int version, int bn, int mt) {
  for (const Variant& v : kVariants)
    if (v.version == version && v.bn == bn && v.mt == mt) return &v;
  return nullptr;
}

// Dispatch (measured on the generator's shapes, batch 32, tools/conv_bench.py; GF_CONV_V2=0 / 1 and GF_CONV_BIG / GF_CONV_MT force):
//   * 16 x 16 patches need enough tiles to fill the GPU: fewer than one per SM -> version 1 with 8 x 16 patches (res 16: 0.056 ms,
//     cuDNN 0.056)
//   * Cin >= 512 with plenty of tiles -> version 1 with 256 x 256 tiles (res 64: 0.702 ms = 881 TFLOP/s, cuDNN 0.698)
//   * everything else -> version 2, shared filter-column boxes (res 32: 0.193 ms vs cuDNN 0.199; res 128: 0.721 vs 0.739;
//     res 256: 0.831 vs 0.781)
static const Variant* dispatch(int B, int H, int W, int Cin, int Cout) {
  static const int v2env = []() { const char* e = getenv("GF_CONV_V2"); return e ? atoi(e) : -1; }();
  const int nsm = num_sms();
  const long long t2 = H % 16 == 0 ? (long long)B * (H / 16) * (W / 16) * (Cout / (Cout % 256 == 0 ? 256 : (Cout % 128 == 0 ? 128 : 64))) : 0;
  const bool big_v1 = Cout % 256 == 0 && Cin >= 512 && t2 >= 4ll * nsm;
  const bool use_v2 = v2env >= 0 ? v2env != 0 : (t2 >= nsm && !big_v1);
  if (use_v2) {
    const bool m2 = H % 16 == 0;
    if (Cout % 256 == 0) return find_variant(2, 256, (m2 && v2env != 2) ? 2 : 1);
    return find_variant(2, Cout % 128 == 0 ? 128 : 64, m2 ? 2 : 1);
  }
  static const int force_mt = []() { const char* e = getenv("GF_CONV_MT"); return e ? atoi(e) : 0; }();     // tuning aid, read once
  const bool mt2 = (H % 16 == 0) && force_mt != 1 && t2 >= nsm;
  static const int big_env = []() { const char* e = getenv("GF_CONV_BIG"); return e ? atoi(e) : -1; }();
  const bool big = big_env >= 0 ? big_env != 0 : big_v1;
  if (Cout % 256 == 0 && big && H % 16 == 0) return find_variant(1, 256, 2);
  if (Cout % 256 == 0 && force_mt != 2) return find_variant(1, 256, 1);
  return find_variant(1, Cout % 128 == 0 ? 128 : 64, mt2 ? 2 : 1);
}

// w [Cout][Cin][3][3] (PyTorch layout) -> wt [9][Cout][Cin], rounded to the nearest TF32
__global__ void pack_weights_kernel(const float* __restrict__ w, float* __restrict__ wt, int Cout, int Cin, float scale) {
  const size_t total = (size_t)9 * Cout * Cin;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin);
    const int o = (int)((i / Cin) % Cout);
    const int tap = (int)(i / ((size_t)Cin * Cout));
    wt[i] = round_tf32_rn(w[((size_t)o * Cin + ci) * 9 + tap] * scale);
  }
}

}  // namespace cv
}  // namespace gf

using namespace gf;

extern "C" int gf_conv3x3_pack_weights(const float* w, float* wt, int Cout, int Cin, float scale, void* stream) {
  if (!w || !wt || Cout <= 0 || Cin <= 0) { set_error("gf_conv3x3_pack_weights: bad arguments"); return GF_ERR_INVALID; }
  const size_t total = (size_t)9 * Cout * Cin;
  size_t blocks = (total + 255) / 256;
  if (blocks > (size_t)num_sms() * 16) blocks = (size_t)num_sms() * 16;
  cv::pack_weights_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(w, wt, Cout, Cin, scale);
  GF_LAUNCH_OK();
  return GF_OK;
}

static thread_local int g_last_variant[3] = {0, 0, 0};      // (version, bn, mt) the last call on this thread launched, zeros if none

extern "C" int gf_conv3x3_nhwc_tf32_ex(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout,
                                       int version, int bn, int mt, void* stream) {
  g_last_variant[0] = g_last_variant[1] = g_last_variant[2] = 0;
  if (!x || !wt || !y) { set_error("gf_conv3x3_nhwc_tf32: null pointer"); return GF_ERR_INVALID; }
  if (B <= 0 || H % cv::PH || W % cv::PW || Cin % cv::BK || Cout % 64 || Cin <= 0 || Cout <= 0) {
    set_error("gf_conv3x3_nhwc_tf32: needs H %% 8 == 0, W %% 16 == 0, Cin %% 32 == 0, Cout %% 64 == 0 (got B=%d H=%d W=%d Cin=%d Cout=%d)", B, H, W, Cin, Cout);
    return GF_ERR_UNSUPPORTED;
  }
  if (((uintptr_t)x & 15) || ((uintptr_t)wt & 15) || ((uintptr_t)y & 15)) { set_error("gf_conv3x3_nhwc_tf32: pointers must be 16-byte aligned"); return GF_ERR_INVALID; }
  const cv::Variant* v = nullptr;
  if (version || bn || mt) {
    if (!(v = cv::find_variant(version, bn, mt))) {
      set_error("gf_conv3x3_nhwc_tf32_ex: no instantiation (version=%d, bn=%d, mt=%d): version 1 or 2, bn 64 / 128 / 256, mt 1 or 2, "
                "or all three 0 for the dispatch", version, bn, mt);
      return GF_ERR_UNSUPPORTED;
    }
    if (Cout % bn || H % (cv::PH * mt)) {
      set_error("gf_conv3x3_nhwc_tf32_ex: (version=%d, bn=%d, mt=%d) needs Cout %% %d == 0 and H %% %d == 0 (got Cout=%d H=%d)",
                version, bn, mt, bn, cv::PH * mt, Cout, H);
      return GF_ERR_UNSUPPORTED;
    }
  }
  int rc;
  if ((rc = check_device())) return rc;
  if (!v) v = cv::dispatch(B, H, W, Cin, Cout);
  if ((rc = v->fn(x, wt, y, B, H, W, Cin, Cout, (cudaStream_t)stream))) return rc;
  g_last_variant[0] = v->version; g_last_variant[1] = v->bn; g_last_variant[2] = v->mt;
  return GF_OK;
}

extern "C" int gf_conv3x3_nhwc_tf32(const float* x, const float* wt, float* y, int B, int H, int W, int Cin, int Cout, void* stream) {
  return gf_conv3x3_nhwc_tf32_ex(x, wt, y, B, H, W, Cin, Cout, 0, 0, 0, stream);
}

extern "C" int gf_conv3x3_last_variant(int* version, int* bn, int* mt) {
  if (!version || !bn || !mt) { set_error("gf_conv3x3_last_variant: null pointer"); return GF_ERR_INVALID; }
  *version = g_last_variant[0]; *bn = g_last_variant[1]; *mt = g_last_variant[2];
  return GF_OK;
}
