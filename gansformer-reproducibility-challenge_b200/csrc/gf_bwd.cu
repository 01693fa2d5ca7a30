// gf_bwd.cu -- backward of stage T (SURVEY row f2): the per-token part of d(loss)/d(x, K', V^T, Rt, Ct).
//
// Forward (oracle/folded.py per_token):  s = x.K'^T + Rt[h] + Ct[w];  p = softmax(s);  ctl = p.V^T (gain | bias);
//     xn = LayerNorm(x) (or x);   out = xn*g  |  xn + g  |  xn*g + b.
// Given dOut this kernel recomputes s, p and the statistics and writes, in three sweeps over the 32-channel chunks of a
// 128-token tile (thread = token, fp32 FMA):
//     dX   [B,n,C]     = LN^T(dxn) + ds.K'                      (the activation gradient)
//     dS   [B,n,KP]    = p * (dp - <p, dp>),  dp = dCtl.V^T     (gradient w.r.t. the logits)
//     P    [B,n,KP]    the probabilities
//     dCtl [B,n,Cout]  = dOut*xn (gain half) | dOut (bias half) (gradient w.r.t. the control signal)
// The remaining reductions over tokens are plain batched GEMMs / sums done by the caller (autograd.py):
//     dK'[b] = dS[b]^T X[b],   dV^T[b] = dCtl[b]^T P[b],   dRt = sum_w dS,   dCt = sum_h dS,
// and the chain rule through stages I and W is torch autograd over tiny [B,k,*] tensors.
// Replaces ~45 full passes over [B,n,C]-sized tensors of the direct-form autograd composite by 8.
//
// Backward of duplex pass A (the centroid softmax over the n grid cells), per image, latent j < k, token t:
//     Sa[j,t] = x_t.M_j + Rt2[h(t),j] + Ct2[w(t),j],   A = softmax_t(Sa),   Xbar = A X.
// gf_attn_centroid_recompute re-runs the pass-A kernel of gf_simt.cu on the caller's fp32 tables (Xbar and lse_j =
// log sum_t exp Sa[j,t]); centroid_bwd_kernel then, given dXbar, streams the tokens once more (thread = token, two sweeps over
// the 32-channel chunks):
//     A[j,t] = exp(Sa - lse_j),  dA = x_t.dXbar_j,  r_j = Xbar_j.dXbar_j,  dSa = A (dA - r),
//     dX += dSa.M + A.dXbar   (accumulated onto the stage-T activation gradient: no extra full-size pass)
// and writes dSa [B,n,KP]; the caller reduces dM = dSa^T X, dRt2 = sum_w dSa, dCt2 = sum_h dSa.
#include <string.h>
#include "gf_common.cuh"

namespace gf {

static constexpr int BTM = 128;     // tokens per CTA (one thread per token)
static constexpr int BCH = 32;      // channels per chunk
static constexpr int BXS = BCH + 4; // padded smem row

struct BwdParams {
  const float* X; const float* dOut; const float* Kp; const float* Vt; const float* Rt; const float* Ct;
  float* dX; float* dS; float* P; float* dCtl;
  int n, H, W, C, k, Cout, norm, integration;
  DropoutArgs dp;            // attention dropout of the forward call (thr = 0: off)
  const float* cb;           // [Cout] bo (+1): ctl = sum_j q_j (Vt_j - cb) + cb when dropout is on
};

__device__ __forceinline__ void bwd_load_chunk(float (*dst)[BXS], const float* __restrict__ src, int t0, int n, int ld, int c0) {
#pragma unroll
  for (int it = 0; it < BTM / 16; ++it) {
    const int row = it * 16 + (threadIdx.x >> 3), c4 = (threadIdx.x & 7) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t0 + row < n) v = __ldg(reinterpret_cast<const float4*>(src + (size_t)(t0 + row) * ld + c0 + c4));
    *reinterpret_cast<float4*>(&dst[row][c4]) = v;
  }
}
__device__ __forceinline__ void bwd_store_chunk(float* __restrict__ dst, float (*src)[BXS], int t0, int n, int ld, int c0) {
#pragma unroll
  for (int it = 0; it < BTM / 16; ++it) {
    const int row = it * 16 + (threadIdx.x >> 3), c4 = (threadIdx.x & 7) * 4;
    if (t0 + row < n) *reinterpret_cast<float4*>(dst + (size_t)(t0 + row) * ld + c0 + c4) = *reinterpret_cast<const float4*>(&src[row][c4]);
  }
}

template <int KP>
__global__ void __launch_bounds__(BTM) token_bwd_kernel(const BwdParams P) {
  extern __shared__ __align__(16) uint8_t bsm_raw[];
  float (*xs)[BXS] = reinterpret_cast<float (*)[BXS]>(bsm_raw);                               // x chunk / result staging
  float (*gs)[BXS] = reinterpret_cast<float (*)[BXS]>(bsm_raw + sizeof(float) * BTM * BXS);   // dOut chunk / dCtl staging
  float (*ks)[BCH] = reinterpret_cast<float (*)[BCH]>(bsm_raw + 2 * sizeof(float) * BTM * BXS);         // K' chunk [KP][32]
  float (*vs)[KP] = reinterpret_cast<float (*)[KP]>(reinterpret_cast<uint8_t*>(ks) + sizeof(float) * KP * BCH);   // V^T gain chunk [32][KP]
  float (*vs2)[KP] = reinterpret_cast<float (*)[KP]>(reinterpret_cast<uint8_t*>(vs) + sizeof(float) * KP * BCH);   // V^T bias chunk

  const int b = blockIdx.y, t0 = blockIdx.x * BTM, tid = threadIdx.x, t = t0 + tid;
  const int n = P.n, C = P.C, Cout = P.Cout, integ = P.integration;
  const bool valid = t < n;
  const float* Xb = P.X + (size_t)b * n * C;
  const float* Gb = P.dOut + (size_t)b * n * C;
  const float* Kpb = P.Kp + (size_t)b * KP * C;
  const float* Vtb = P.Vt + (size_t)b * Cout * KP;
  float* dXb = P.dX + (size_t)b * n * C;
  float* dCb = P.dCtl + (size_t)b * n * Cout;

  float s[KP];
  {
    const int h = valid ? t / P.W : 0, w = valid ? t % P.W : 0;
    const float* rt = P.Rt + ((size_t)b * P.H + h) * KP;
    const float* ct = P.Ct + ((size_t)b * P.W + w) * KP;
#pragma unroll
    for (int j = 0; j < KP; ++j) s[j] = rt[j] + ct[j];
  }
  // ---- sweep 1: logits + layer-norm statistics (as the forward)
  float sum = 0.f, sumsq = 0.f, shift = 0.f;
  for (int c0 = 0; c0 < C; c0 += BCH) {
    __syncthreads();
    bwd_load_chunk(xs, Xb, t0, n, C, c0);
    for (int i = tid; i < KP * BCH / 4; i += BTM) {
      const int j = i / (BCH / 4), c4 = (i % (BCH / 4)) * 4;
      *reinterpret_cast<float4*>(&ks[j][c4]) = __ldg(reinterpret_cast<const float4*>(Kpb + (size_t)j * C + c0 + c4));
    }
    __syncthreads();
    if (c0 == 0) shift = xs[tid][0];
#pragma unroll
    for (int c4 = 0; c4 < BCH; c4 += 4) {
      const float4 x = *reinterpret_cast<const float4*>(&xs[tid][c4]);
      const float d0 = x.x - shift, d1 = x.y - shift, d2 = x.z - shift, d3 = x.w - shift;
      sum += (d0 + d1) + (d2 + d3);
      sumsq = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, sumsq))));
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        const float4 kv = *reinterpret_cast<const float4*>(&ks[j][c4]);
        s[j] = fmaf(x.x, kv.x, fmaf(x.y, kv.y, fmaf(x.z, kv.z, fmaf(x.w, kv.w, s[j]))));
      }
    }
  }
  float mx = s[0];
#pragma unroll
  for (int j = 1; j < KP; ++j) mx = fmaxf(mx, s[j]);
  float den = 0.f;
#pragma unroll
  for (int j = 0; j < KP; ++j) { s[j] = expf(s[j] - mx); den += s[j]; }
  const float inv = 1.f / den;
#pragma unroll
  for (int j = 0; j < KP; ++j) s[j] *= inv;                       // s = p from here on
  // attention dropout: q = p * mk feeds the control signal (and the dV^T reduction); the softmax backward uses p itself
  float pk[KP];                                                  // p before dropout (only read when dropout is on)
  float mk[KP];
#pragma unroll
  for (int j = 0; j < KP; ++j) { pk[j] = s[j]; mk[j] = 1.f; }
  if (P.dp.thr) {
    const unsigned long long seed = P.dp.state[0], step = P.dp.state[1];
#pragma unroll
    for (int q = 0; q < KP / 4; ++q) {
      dropout_mult4(P.dp, seed, step, (uint32_t)((size_t)b * n + (valid ? t : 0)), q, mk + q * 4);
      s[q * 4] *= mk[q * 4]; s[q * 4 + 1] *= mk[q * 4 + 1]; s[q * 4 + 2] *= mk[q * 4 + 2]; s[q * 4 + 3] *= mk[q * 4 + 3];
    }
  }                                                              // s = q (= p without dropout) from here on
  float qdef = 0.f;                                              // 1 - sum q (0 without dropout)
  if (P.dp.thr) {
    float qs = 0.f;
#pragma unroll
    for (int j = 0; j < KP; ++j) qs += s[j];
    qdef = 1.f - qs;
  }
  float dcb = 0.f;                                               // sum_c dctl[c] * cb[c]: d/dq_j of the (1 - sum q) cb term is -cb
  float mean = 0.f, rstd = 1.f;
  const bool ln = P.norm == GF_NORM_LAYER;
  if (ln) {
    const float invC = 1.f / (float)C;
    const float md = sum * invC;
    const float var = fmaxf(sumsq * invC - md * md, 0.f);
    mean = md + shift;
    rstd = rsqrtf(var + 1e-8f);
  }

  // ---- sweep 2: dCtl (stored), dp, and the two LayerNorm-backward sums
  float dp[KP];
#pragma unroll
  for (int j = 0; j < KP; ++j) dp[j] = 0.f;
  float a1 = 0.f, a2 = 0.f;                                      // sum_c dxn, sum_c dxn * xn
  for (int c0 = 0; c0 < C; c0 += BCH) {
    __syncthreads();
    bwd_load_chunk(xs, Xb, t0, n, C, c0);
    bwd_load_chunk(gs, Gb, t0, n, C, c0);
    for (int i = tid; i < BCH * KP / 4; i += BTM)
      reinterpret_cast<float4*>(&vs[0][0])[i] = __ldg(reinterpret_cast<const float4*>(Vtb + (size_t)c0 * KP) + i);
    if (integ == GF_INT_BOTH)
      for (int i = tid; i < BCH * KP / 4; i += BTM)
        reinterpret_cast<float4*>(&vs2[0][0])[i] = __ldg(reinterpret_cast<const float4*>(Vtb + (size_t)(C + c0) * KP) + i);
    __syncthreads();
    if (integ == GF_INT_BOTH) bwd_store_chunk(dCb, gs, t0, n, Cout, C + c0);      // bias half of dCtl = dOut (before gs is reused)
    __syncthreads();
#pragma unroll 2
    for (int cc = 0; cc < BCH; ++cc) {
      const float go = gs[tid][cc];
      const float xn = (xs[tid][cc] - mean) * rstd;
      float dxn, dc;
      if (integ == GF_INT_ADD) { dxn = go; dc = go; }
      else {
        float g = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < KP; j4 += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&vs[cc][j4]);
          g = fmaf(s[j4], v.x, fmaf(s[j4 + 1], v.y, fmaf(s[j4 + 2], v.z, fmaf(s[j4 + 3], v.w, g))));
        }
        if (P.dp.thr) g = fmaf(qdef, __ldg(P.cb + c0 + cc), g);
        dxn = go * g; dc = go * xn;
      }
      if (P.dp.thr) {
        dcb = fmaf(dc, __ldg(P.cb + c0 + cc), dcb);
        if (integ == GF_INT_BOTH) dcb = fmaf(go, __ldg(P.cb + C + c0 + cc), dcb);
      }
      a1 += dxn; a2 = fmaf(dxn, xn, a2);
#pragma unroll
      for (int j4 = 0; j4 < KP; j4 += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&vs[cc][j4]);
        dp[j4] = fmaf(dc, v.x, dp[j4]); dp[j4 + 1] = fmaf(dc, v.y, dp[j4 + 1]);
        dp[j4 + 2] = fmaf(dc, v.z, dp[j4 + 2]); dp[j4 + 3] = fmaf(dc, v.w, dp[j4 + 3]);
      }
      if (integ == GF_INT_BOTH) {
#pragma unroll
        for (int j4 = 0; j4 < KP; j4 += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&vs2[cc][j4]);
          dp[j4] = fmaf(go, v.x, dp[j4]); dp[j4 + 1] = fmaf(go, v.y, dp[j4 + 1]);
          dp[j4 + 2] = fmaf(go, v.z, dp[j4 + 2]); dp[j4 + 3] = fmaf(go, v.w, dp[j4 + 3]);
        }
      }
      gs[tid][cc] = dc;                                          // own row only: no hazard with other threads
    }
    __syncthreads();
    bwd_store_chunk(dCb, gs, t0, n, Cout, c0);                    // gain half (or the only half) of dCtl
  }
  // ---- softmax backward; dS and P rows
  float pd = 0.f;
#pragma unroll
  for (int j = 0; j < KP; ++j) { dp[j] = (dp[j] - dcb) * mk[j]; pd = fmaf(pk[j], dp[j], pd); }   // d/dq (minus the cb term) -> d/dp through the mask
#pragma unroll
  for (int j = 0; j < KP; ++j) dp[j] = pk[j] * (dp[j] - pd);     // dp = ds from here on
  if (valid) {
    float4* ds4 = reinterpret_cast<float4*>(P.dS + ((size_t)b * n + t) * KP);
    float4* p4 = reinterpret_cast<float4*>(P.P + ((size_t)b * n + t) * KP);
#pragma unroll
    for (int j4 = 0; j4 < KP / 4; ++j4) {
      ds4[j4] = make_float4(dp[j4 * 4], dp[j4 * 4 + 1], dp[j4 * 4 + 2], dp[j4 * 4 + 3]);
      p4[j4] = make_float4(s[j4 * 4], s[j4 * 4 + 1], s[j4 * 4 + 2], s[j4 * 4 + 3]);
    }
  }
  const float m1 = a1 / (float)C, m2 = a2 / (float)C;

  // ---- sweep 3: dX = LayerNorm^T(dxn) + ds.K'
  for (int c0 = 0; c0 < C; c0 += BCH) {
    __syncthreads();
    bwd_load_chunk(xs, Xb, t0, n, C, c0);
    bwd_load_chunk(gs, Gb, t0, n, C, c0);
    for (int i = tid; i < KP * BCH / 4; i += BTM) {
      const int j = i / (BCH / 4), c4 = (i % (BCH / 4)) * 4;
      *reinterpret_cast<float4*>(&ks[j][c4]) = __ldg(reinterpret_cast<const float4*>(Kpb + (size_t)j * C + c0 + c4));
    }
    if (integ != GF_INT_ADD)
      for (int i = tid; i < BCH * KP / 4; i += BTM)
        reinterpret_cast<float4*>(&vs[0][0])[i] = __ldg(reinterpret_cast<const float4*>(Vtb + (size_t)c0 * KP) + i);
    __syncthreads();
#pragma unroll 2
    for (int cc = 0; cc < BCH; ++cc) {
      const float go = gs[tid][cc];
      float dxn = go;
      if (integ != GF_INT_ADD) {
        float g = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < KP; j4 += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&vs[cc][j4]);
          g = fmaf(s[j4], v.x, fmaf(s[j4 + 1], v.y, fmaf(s[j4 + 2], v.z, fmaf(s[j4 + 3], v.w, g))));
        }
        if (P.dp.thr) g = fmaf(qdef, __ldg(P.cb + c0 + cc), g);
        dxn = go * g;
      }
      float dx = dxn;
      if (ln) {
        const float xn = (xs[tid][cc] - mean) * rstd;
        dx = rstd * (dxn - m1 - xn * m2);
      }
#pragma unroll
      for (int j = 0; j < KP; ++j) dx = fmaf(dp[j], ks[j][cc], dx);
      xs[tid][cc] = dx;
    }
    __syncthreads();
    bwd_store_chunk(dXb, xs, t0, n, C, c0);
  }
}

struct CenBwdParams {
  const float* X; const float* M; const float* Rt; const float* Ct; const float* lse; const float* Xbar; const float* dXbar;
  float* dX; float* dSa;
  int n, H, W, C, k;
};

// M / dXbar chunk [KP][32] of image b; rows j >= k are zero, so the padded latents contribute exactly nothing
template <int KP>
__device__ __forceinline__ void cen_load_tables(float (*ms)[BCH], float (*gs)[BCH], const float* __restrict__ Mb, const float* __restrict__ Gb,
                                                int k, int C, int c0) {
  for (int i = threadIdx.x; i < KP * BCH / 4; i += BTM) {
    const int j = i / (BCH / 4), c4 = (i % (BCH / 4)) * 4;
    float4 m = make_float4(0.f, 0.f, 0.f, 0.f), g = m;
    if (j < k) {
      m = __ldg(reinterpret_cast<const float4*>(Mb + (size_t)j * C + c0 + c4));
      g = __ldg(reinterpret_cast<const float4*>(Gb + (size_t)j * C + c0 + c4));
    }
    *reinterpret_cast<float4*>(&ms[j][c4]) = m;
    *reinterpret_cast<float4*>(&gs[j][c4]) = g;
  }
}

template <int KP>
__global__ void __launch_bounds__(BTM) centroid_bwd_kernel(const CenBwdParams P) {
  __shared__ __align__(16) float xs[BTM][BXS];     // x chunk (sweep 1), dX chunk (sweep 2)
  __shared__ __align__(16) float ms[KP][BCH];      // M chunk
  __shared__ __align__(16) float gs[KP][BCH];      // dXbar chunk
  __shared__ float rs[KP];                         // r_j = Xbar_j . dXbar_j of this image

  const int b = blockIdx.y, t0 = blockIdx.x * BTM, tid = threadIdx.x, t = t0 + tid;
  const int n = P.n, C = P.C, k = P.k;
  const bool valid = t < n;
  const float* Xb = P.X + (size_t)b * n * C;
  const float* Mb = P.M + (size_t)b * KP * C;
  const float* Gb = P.dXbar + (size_t)b * k * C;
  const float* XBb = P.Xbar + (size_t)b * k * C;
  float* dXb = P.dX + (size_t)b * n * C;

  float s[KP], da[KP];
  {
    const int h = valid ? t / P.W : 0, w = valid ? t % P.W : 0;
    const float* rt = P.Rt + ((size_t)b * P.H + h) * KP;
    const float* ct = P.Ct + ((size_t)b * P.W + w) * KP;
#pragma unroll
    for (int j = 0; j < KP; ++j) { s[j] = rt[j] + ct[j]; da[j] = 0.f; }
  }
  float racc = 0.f;                                // thread j < k: its latent's r_j, chunk by chunk
  // ---- sweep 1: logits Sa and dA = x.dXbar
  for (int c0 = 0; c0 < C; c0 += BCH) {
    __syncthreads();
    bwd_load_chunk(xs, Xb, t0, n, C, c0);
    cen_load_tables<KP>(ms, gs, Mb, Gb, k, C, c0);
    __syncthreads();
    if (tid < k) {
#pragma unroll
      for (int c4 = 0; c4 < BCH; c4 += 4) {
        const float4 xb = __ldg(reinterpret_cast<const float4*>(XBb + (size_t)tid * C + c0 + c4));
        const float4 g = *reinterpret_cast<const float4*>(&gs[tid][c4]);
        racc = fmaf(xb.x, g.x, fmaf(xb.y, g.y, fmaf(xb.z, g.z, fmaf(xb.w, g.w, racc))));
      }
    }
#pragma unroll
    for (int c4 = 0; c4 < BCH; c4 += 4) {
      const float4 x = *reinterpret_cast<const float4*>(&xs[tid][c4]);
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        const float4 m = *reinterpret_cast<const float4*>(&ms[j][c4]);
        const float4 g = *reinterpret_cast<const float4*>(&gs[j][c4]);
        s[j] = fmaf(x.x, m.x, fmaf(x.y, m.y, fmaf(x.z, m.z, fmaf(x.w, m.w, s[j]))));
        da[j] = fmaf(x.x, g.x, fmaf(x.y, g.y, fmaf(x.z, g.z, fmaf(x.w, g.w, da[j]))));
      }
    }
  }
  if (tid < KP) rs[tid] = tid < k ? racc : 0.f;
  __syncthreads();
  // ---- A and dSa (s = A, da = dSa from here on); padded latents: exactly 0
  const float* lse = P.lse + (size_t)b * k;
#pragma unroll
  for (int j = 0; j < KP; ++j) {
    float a = 0.f, ds = 0.f;
    if (j < k) {
      a = expf(s[j] - __ldg(lse + j));
      ds = a * (da[j] - rs[j]);
    }
    s[j] = a; da[j] = ds;
  }
  if (valid) {
    float4* ds4 = reinterpret_cast<float4*>(P.dSa + ((size_t)b * n + t) * KP);
#pragma unroll
    for (int j4 = 0; j4 < KP / 4; ++j4) ds4[j4] = make_float4(da[j4 * 4], da[j4 * 4 + 1], da[j4 * 4 + 2], da[j4 * 4 + 3]);
  }
  // ---- sweep 2: dX += dSa.M + A.dXbar
  for (int c0 = 0; c0 < C; c0 += BCH) {
    __syncthreads();
    bwd_load_chunk(xs, dXb, t0, n, C, c0);
    cen_load_tables<KP>(ms, gs, Mb, Gb, k, C, c0);
    __syncthreads();
#pragma unroll
    for (int c4 = 0; c4 < BCH; c4 += 4) {
      float4 acc = *reinterpret_cast<const float4*>(&xs[tid][c4]);
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        const float4 m = *reinterpret_cast<const float4*>(&ms[j][c4]);
        const float4 g = *reinterpret_cast<const float4*>(&gs[j][c4]);
        acc.x = fmaf(da[j], m.x, fmaf(s[j], g.x, acc.x)); acc.y = fmaf(da[j], m.y, fmaf(s[j], g.y, acc.y));
        acc.z = fmaf(da[j], m.z, fmaf(s[j], g.z, acc.z)); acc.w = fmaf(da[j], m.w, fmaf(s[j], g.w, acc.w));
      }
      *reinterpret_cast<float4*>(&xs[tid][c4]) = acc;           // own row only: no hazard with other threads
    }
    __syncthreads();
    bwd_store_chunk(dXb, xs, t0, n, C, c0);
  }
}

// shared checks of the two pass-A entry points: a duplex descriptor (its workspace layout has the pass-A partials), grid limits
static int centroid_entry_layout(const gf_attn_desc* desc, Layout* L, const char* what) {
  int rc = make_layout(desc, L);
  if (rc) return rc;
  if (!L->duplex) { set_error("%s: desc.duplex is 0 (pass A exists in duplex layers only)", what); return GF_ERR_INVALID; }
  if (L->B > 65535) { set_error("%s: B > 65535", what); return GF_ERR_UNSUPPORTED; }
  return GF_OK;
}

}  // namespace gf

using namespace gf;

extern "C" int gf_attn_centroid_recompute(const gf_attn_desc* desc, const float* X, const float* M, const float* Rt2, const float* Ct2,
                                          float* Xbar, float* lse, void* ws, void* stream) {
  Layout L;
  int rc = centroid_entry_layout(desc, &L, "gf_attn_centroid_recompute");
  if (rc) return rc;
  if (!X || !M || !Rt2 || !Ct2 || !Xbar || !lse || !ws) { set_error("gf_attn_centroid_recompute: null pointer"); return GF_ERR_INVALID; }
  if ((rc = check_device())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  if ((rc = centroid_partials_simt(L, X, M, Rt2, Ct2, (float*)ws + L.w_PART, st))) return rc;
  return centroid_merge(L, (float*)ws, st, nullptr, 0, Xbar, lse);
}

extern "C" int gf_attn_centroid_bwd(const gf_attn_desc* desc, const float* X, const float* M, const float* Rt2, const float* Ct2,
                                    const float* lse, const float* Xbar, const float* dXbar, float* dX, float* dSa, void* stream) {
  Layout L;
  int rc = centroid_entry_layout(desc, &L, "gf_attn_centroid_bwd");
  if (rc) return rc;
  if (!X || !M || !Rt2 || !Ct2 || !lse || !Xbar || !dXbar || !dX || !dSa) { set_error("gf_attn_centroid_bwd: null pointer"); return GF_ERR_INVALID; }
  if ((rc = check_device())) return rc;
  CenBwdParams P;
  P.X = X; P.M = M; P.Rt = Rt2; P.Ct = Ct2; P.lse = lse; P.Xbar = Xbar; P.dXbar = dXbar; P.dX = dX; P.dSa = dSa;
  P.n = L.n; P.H = L.H; P.W = L.W; P.C = L.C; P.k = L.k;
  dim3 grid((L.n + BTM - 1) / BTM, L.B);
  cudaStream_t st = (cudaStream_t)stream;
  if (L.KP == 16) centroid_bwd_kernel<16><<<grid, BTM, 0, st>>>(P);
  else centroid_bwd_kernel<32><<<grid, BTM, 0, st>>>(P);
  GF_LAUNCH_OK();
  return GF_OK;
}

extern "C" int gf_attn_simplex_bwd(const gf_attn_desc* desc, const float* X, const float* dOut, const float* Kp, const float* Vt,
                                   const float* Rt, const float* Ct, float* dX, float* dS, float* Pout, float* dCtl, void* stream) {
  return gf_attn_simplex_bwd_ex(desc, X, dOut, Kp, Vt, Rt, Ct, dX, dS, Pout, dCtl, 0.f, 0, nullptr, nullptr, stream);
}

extern "C" int gf_attn_simplex_bwd_ex(const gf_attn_desc* desc, const float* X, const float* dOut, const float* Kp, const float* Vt,
                                      const float* Rt, const float* Ct, float* dX, float* dS, float* Pout, float* dCtl,
                                      float att_dp, uint32_t dp_salt, const unsigned long long* dp_state, const float* cb, void* stream) {
  Layout L;
  int rc = make_layout(desc, &L);
  if (rc) return rc;
  if (!X || !dOut || !Kp || !Vt || !Rt || !Ct || !dX || !dS || !Pout || !dCtl) { set_error("gf_attn_simplex_bwd: null pointer"); return GF_ERR_INVALID; }
  if (L.duplex) { set_error("gf_attn_simplex_bwd: duplex layers use the composite backward"); return GF_ERR_UNSUPPORTED; }
  if (desc->norm != GF_NORM_LAYER && desc->norm != GF_NORM_NONE) { set_error("gf_attn_simplex_bwd: norm must be layer or none"); return GF_ERR_UNSUPPORTED; }
  if (L.B > 65535) { set_error("gf_attn_simplex_bwd: B > 65535"); return GF_ERR_UNSUPPORTED; }
  if ((rc = check_device())) return rc;
  BwdParams P;
  P.X = X; P.dOut = dOut; P.Kp = Kp; P.Vt = Vt; P.Rt = Rt; P.Ct = Ct; P.dX = dX; P.dS = dS; P.P = Pout; P.dCtl = dCtl;
  P.n = L.n; P.H = L.H; P.W = L.W; P.C = L.C; P.k = L.k; P.Cout = L.Cout; P.norm = desc->norm; P.integration = desc->integration;
  {
    gf_attn_postop post;
    memset(&post, 0, sizeof(post));
    post.att_dp = att_dp; post.dp_salt = dp_salt; post.dp_state = dp_state;
    if ((rc = dropout_args(&post, &P.dp))) return rc;
    if (P.dp.thr && !cb) { set_error("gf_attn_simplex_bwd_ex: attention dropout needs cb (bo, +1 on the gain half)"); return GF_ERR_INVALID; }
    P.cb = cb;
  }
  if (L.heads != 1) { set_error("gf_attn_simplex_bwd: one head (multi-head layers use the composite backward)"); return GF_ERR_UNSUPPORTED; }
  dim3 grid((L.n + BTM - 1) / BTM, L.B);
  const int smem = (int)(2 * sizeof(float) * BTM * BXS + 3 * sizeof(float) * L.KP * BCH);
  cudaStream_t st = (cudaStream_t)stream;
  if (L.KP == 16) {
    GF_CUDA_OK(cudaFuncSetAttribute(token_bwd_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    token_bwd_kernel<16><<<grid, BTM, smem, st>>>(P);
  } else {
    GF_CUDA_OK(cudaFuncSetAttribute(token_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    token_bwd_kernel<32><<<grid, BTM, smem, st>>>(P);
  }
  GF_LAUNCH_OK();
  return GF_OK;
}
