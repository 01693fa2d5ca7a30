// gf_simt.cu -- CUDA-core fp32-FMA kernels of stage T (tight-tolerance mode and shapes the tcgen05 kernel
// does not take), the instance/batch-norm statistics pass, and duplex pass A (centroids).
//
// Replaces, on the reference side (expected src/training/network.py, not in the checkout): the body of
// transformer_layer (Q projection, QK^T, softmax, PV), integrate and att_norm.  Algorithm = oracle/folded.py
// per_token() / centroid_pass().
#include "gf_common.cuh"

namespace gf {

static constexpr int TM = 128;      // tokens per CTA (one thread per token)
static constexpr int CH = 32;       // channels per smem chunk
static constexpr int XS = CH + 4;   // padded smem row (144 B: LDS.128 by row is conflict-free)

struct TokenParams {
  const float* X; float* Xout; float* att;
  const float* Kp; const float* Vt; const float* Rt; const float* Ct;
  const float* nscale; const float* nshift;
  int n, H, W, C, k, Cout;
  int norm, integration;
  // fused epilogue (gf_attn_postop)
  const float* pbias; const float* pnoise; const float* pstrength; long long pnoise_bstride; int pact; float pgain; int has_post;
  const float* in_scale; const float* post_scale; int in_ld, post_ld;
  int heads, seg;            // multi-head: softmax per segment of `seg` table columns (heads * seg == KP)
  DropoutArgs dp;            // attention dropout (training): thr = 0 when off
  const float* cb;           // [Cout] bo (+1): re-added as (1 - sum q) * cb when the mask broke sum q = 1
};

__device__ __forceinline__ void load_x_chunk(float (*xs)[XS], const float* __restrict__ Xb, int t0, int n, int C, int c0) {
  // 128 tokens x 32 channels, float4 per thread, 8 threads per row -> each row is one coalesced 128 B line
#pragma unroll
  for (int it = 0; it < TM / 16; ++it) {
    const int row = it * 16 + (threadIdx.x >> 3), c4 = (threadIdx.x & 7) * 4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (t0 + row < n) v = __ldg(reinterpret_cast<const float4*>(Xb + (size_t)(t0 + row) * C + c0 + c4));
    *reinterpret_cast<float4*>(&xs[row][c4]) = v;
  }
}

template <int KP>
__global__ void __launch_bounds__(TM) token_simt_kernel(const TokenParams P) {
  __shared__ __align__(16) float xs[TM][XS];
  __shared__ __align__(16) float ks[KP][CH];        // K' chunk, later reused for V^T chunks [CH][KP] (gain)
  __shared__ __align__(16) float vs2[CH][KP];       // bias half of V^T ("both")
  __shared__ float nsc[CH], nsh[CH], pbs[CH], isc[CH], psc[CH];

  const int b = blockIdx.y, t0 = blockIdx.x * TM, tid = threadIdx.x, t = t0 + tid;
  const int n = P.n, C = P.C;
  const bool valid = t < n;
  const float* Xb = P.X + (size_t)b * n * C;
  float* Ob = P.Xout + (size_t)b * n * C;
  const float* Kpb = P.Kp + (size_t)b * KP * C;
  const float* Vtb = P.Vt + (size_t)b * P.Cout * KP;

  float s[KP];
  {
    const int h = valid ? t / P.W : 0, w = valid ? t % P.W : 0;
    const float* rt = P.Rt + ((size_t)b * P.H + h) * KP;
    const float* ct = P.Ct + ((size_t)b * P.W + w) * KP;
#pragma unroll
    for (int j = 0; j < KP; ++j) s[j] = rt[j] + ct[j];
  }

  // ---- sweep 1: logits + layer-norm statistics ------------------------------------------------------
  float sum = 0.f, sumsq = 0.f, shift = 0.f;
  for (int c0 = 0; c0 < C; c0 += CH) {
    __syncthreads();
    load_x_chunk(xs, Xb, t0, n, C, c0);
    for (int i = tid; i < KP * CH / 4; i += TM) {
      const int j = i / (CH / 4), c4 = (i % (CH / 4)) * 4;
      *reinterpret_cast<float4*>(&ks[j][c4]) = __ldg(reinterpret_cast<const float4*>(Kpb + (size_t)j * C + c0 + c4));
    }
    if (tid < CH) isc[tid] = P.in_scale ? P.in_scale[(size_t)b * P.in_ld + c0 + tid] : 1.f;
    __syncthreads();
    if (c0 == 0) shift = xs[tid][0] * isc[0];   // shifted sums: avoids cancellation in E[x^2]-E[x]^2
#pragma unroll
    for (int c4 = 0; c4 < CH; c4 += 4) {
      const float4 xr = *reinterpret_cast<const float4*>(&xs[tid][c4]);
      const float4 xq = make_float4(xr.x * isc[c4], xr.y * isc[c4 + 1], xr.z * isc[c4 + 2], xr.w * isc[c4 + 3]);   // statistics see x_in
      const float4 x = xr;                                                                                        // logits: K' already carries in_scale
      const float d0 = xq.x - shift, d1 = xq.y - shift, d2 = xq.z - shift, d3 = xq.w - shift;
      sum += (d0 + d1) + (d2 + d3);
      sumsq = fmaf(d0, d0, fmaf(d1, d1, fmaf(d2, d2, fmaf(d3, d3, sumsq))));
#pragma unroll
      for (int j = 0; j < KP; ++j) {
        const float4 kv = *reinterpret_cast<const float4*>(&ks[j][c4]);
        s[j] = fmaf(x.x, kv.x, fmaf(x.y, kv.y, fmaf(x.z, kv.z, fmaf(x.w, kv.w, s[j]))));
      }
    }
  }

  // ---- softmax over the k latents (padded latents carry -inf from Rt) ------------------------------
  if (P.heads == 1) {
    float mx = s[0];
#pragma unroll
    for (int j = 1; j < KP; ++j) mx = fmaxf(mx, s[j]);
    float den = 0.f;
#pragma unroll
    for (int j = 0; j < KP; ++j) { s[j] = expf(s[j] - mx); den += s[j]; }
    const float inv = 1.f / den;
#pragma unroll
    for (int j = 0; j < KP; ++j) s[j] *= inv;
    if (P.att && valid) {
      float* a = P.att + ((size_t)b * n + t) * P.k;
#pragma unroll
      for (int j = 0; j < KP; ++j) if (j < P.k) a[j] = s[j];
    }
  } else {
    // multi-head: one softmax per head (column segment); attention map = mean over the heads
    const int seg = P.seg;
    float mxs[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY}, dens[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < KP; ++j) { const int g_ = j / seg; mxs[g_] = fmaxf(mxs[g_], s[j]); }
#pragma unroll
    for (int j = 0; j < KP; ++j) { const int g_ = j / seg; s[j] = expf(s[j] - mxs[g_]); dens[g_] += s[j]; }
#pragma unroll
    for (int j = 0; j < KP; ++j) s[j] /= dens[j / seg];
    if (P.att && valid) {
      float* a = P.att + ((size_t)b * n + t) * P.k;
      for (int j = 0; j < P.k; ++j) {
        float m = 0.f;
#pragma unroll
        for (int c = 0; c < KP; ++c) if (c % seg == j) m += s[c];
        a[j] = m / (float)P.heads;
      }
    }
  }

  float qdef = 0.f;          // 1 - sum of the (dropped, rescaled) probabilities: weight of the un-droppable constants
  if (P.dp.thr) {            // attention dropout: drop / rescale the probabilities (the attention map above is pre-dropout)
    const unsigned long long seed = P.dp.state[0], step = P.dp.state[1];
    float qs = 0.f;
#pragma unroll
    for (int q = 0; q < KP / 4; ++q) {
      float mk[4];
      dropout_mult4(P.dp, seed, step, (uint32_t)((size_t)b * n + (valid ? t : 0)), q, mk);
      s[q * 4] *= mk[0]; s[q * 4 + 1] *= mk[1]; s[q * 4 + 2] *= mk[2]; s[q * 4 + 3] *= mk[3];
      qs += (s[q * 4] + s[q * 4 + 1]) + (s[q * 4 + 2] + s[q * 4 + 3]);
    }
    qdef = 1.f - qs;
  }

  float mean = 0.f, rstd = 1.f;
  if (P.norm == GF_NORM_LAYER) {
    const float invC = 1.f / (float)C;
    const float md = sum * invC;                       // mean of (x - shift)
    const float var = fmaxf(sumsq * invC - md * md, 0.f);
    mean = md + shift;
    rstd = rsqrtf(var + 1e-8f);
  }
  const bool affine = P.norm == GF_NORM_INSTANCE || P.norm == GF_NORM_BATCH;
  const int integ = P.integration;
  float pnz = 0.f;
  if (P.has_post && P.pnoise && valid)
    pnz = __ldg(P.pnoise + (size_t)b * P.pnoise_bstride + t) * (P.pstrength ? __ldg(P.pstrength) : 1.f);
  float (*vs)[KP] = reinterpret_cast<float (*)[KP]>(&ks[0][0]);   // [CH][KP] view of the same bytes

  // ---- sweep 2: control signal, normalise, modulate, store -----------------------------------------
  for (int c0 = 0; c0 < C; c0 += CH) {
    __syncthreads();
    load_x_chunk(xs, Xb, t0, n, C, c0);
    for (int i = tid; i < CH * KP / 4; i += TM)
      reinterpret_cast<float4*>(&vs[0][0])[i] = __ldg(reinterpret_cast<const float4*>(Vtb + (size_t)c0 * KP) + i);
    if (integ == GF_INT_BOTH)
      for (int i = tid; i < CH * KP / 4; i += TM)
        reinterpret_cast<float4*>(&vs2[0][0])[i] = __ldg(reinterpret_cast<const float4*>(Vtb + (size_t)(C + c0) * KP) + i);
    if (affine && tid < CH) {
      nsc[tid] = P.nscale[(size_t)b * C + c0 + tid];
      nsh[tid] = P.nshift[(size_t)b * C + c0 + tid];
    }
    if (P.has_post && tid < CH) pbs[tid] = P.pbias ? P.pbias[c0 + tid] : 0.f;
    if (tid < CH) {
      isc[tid] = P.in_scale ? P.in_scale[(size_t)b * P.in_ld + c0 + tid] : 1.f;
      psc[tid] = P.post_scale ? P.post_scale[(size_t)b * P.post_ld + c0 + tid] : 1.f;
    }
    __syncthreads();
#pragma unroll 4
    for (int cc = 0; cc < CH; ++cc) {
      float g = 0.f;
#pragma unroll
      for (int j4 = 0; j4 < KP; j4 += 4) {
        const float4 v = *reinterpret_cast<const float4*>(&vs[cc][j4]);
        g = fmaf(s[j4], v.x, fmaf(s[j4 + 1], v.y, fmaf(s[j4 + 2], v.z, fmaf(s[j4 + 3], v.w, g))));
      }
      if (P.dp.thr) g = fmaf(qdef, __ldg(P.cb + c0 + cc), g);      // the constants (bo, the 1 of 1 + gain) are not dropped
      const float x = xs[tid][cc] * isc[cc];
      float xn;
      if (affine) xn = fmaf(x, nsc[cc], nsh[cc]);
      else xn = (x - mean) * rstd;
      float y;
      if (integ == GF_INT_MUL) y = xn * g;
      else if (integ == GF_INT_ADD) y = xn + g;
      else {
        float bb = 0.f;
#pragma unroll
        for (int j4 = 0; j4 < KP; j4 += 4) {
          const float4 v = *reinterpret_cast<const float4*>(&vs2[cc][j4]);
          bb = fmaf(s[j4], v.x, fmaf(s[j4 + 1], v.y, fmaf(s[j4 + 2], v.z, fmaf(s[j4 + 3], v.w, bb))));
        }
        if (P.dp.thr) bb = fmaf(qdef, __ldg(P.cb + C + c0 + cc), bb);
        y = fmaf(xn, g, bb);
      }
      if (P.has_post) {
        y += pnz + pbs[cc];
        if (P.pact == 1) y = fmaxf(y, 0.2f * y);
        y *= P.pgain * psc[cc];
      }
      xs[tid][cc] = y;
    }
    __syncthreads();
#pragma unroll
    for (int it = 0; it < TM / 16; ++it) {
      const int row = it * 16 + (tid >> 3), c4 = (tid & 7) * 4;
      if (t0 + row < n)
        *reinterpret_cast<float4*>(Ob + (size_t)(t0 + row) * C + c0 + c4) = *reinterpret_cast<const float4*>(&xs[row][c4]);
    }
  }
}

int token_pass_simt(const Layout& L, const gf_attn_desc* d, const float* X, float* Xout, float* att, float* ws, const gf_attn_postop* post, cudaStream_t st) {
  TokenParams P;
  P.X = X; P.Xout = Xout; P.att = att;
  P.Kp = ws + L.w_Kp; P.Vt = ws + L.w_Vt; P.Rt = ws + L.w_Rt; P.Ct = ws + L.w_Ct;
  P.nscale = ws + L.w_NSCALE; P.nshift = ws + L.w_NSHIFT;
  P.n = L.n; P.H = L.H; P.W = L.W; P.C = L.C; P.k = L.k; P.Cout = L.Cout;
  P.norm = d->norm; P.integration = d->integration;
  P.has_post = post ? 1 : 0;
  P.pbias = post ? post->bias : nullptr; P.pnoise = post ? post->noise : nullptr; P.pstrength = post ? post->strength : nullptr;
  P.pnoise_bstride = post ? post->noise_bstride : 0; P.pact = post ? post->act : 0; P.pgain = post ? post->gain : 1.f;
  P.in_scale = post ? post->in_scale : nullptr; P.post_scale = post ? post->post_scale : nullptr;
  P.in_ld = post ? post->in_scale_ld : 0; P.post_ld = post ? post->post_scale_ld : 0;
  P.heads = L.heads; P.seg = L.seg;
  { int rcd = dropout_args(post, &P.dp); if (rcd) return rcd; }
  P.cb = ws + L.w_CB;
  dim3 grid((L.n + TM - 1) / TM, L.B);
  if (L.KP == 16) token_simt_kernel<16><<<grid, TM, 0, st>>>(P);
  else token_simt_kernel<32><<<grid, TM, 0, st>>>(P);
  GF_LAUNCH_OK();
  set_path(GF_PATH_SIMT_FP32);
  return GF_OK;
}

// ------------------------------------------------------------------------------------------------------
// instance / batch norm statistics: per-(b,c) scale = rstd, shift = -mean*rstd
// ------------------------------------------------------------------------------------------------------
// grid (nsplit, B), block = 256 threads = 8 token lanes x 32 channel lanes; loops channel groups of 32.
__global__ void __launch_bounds__(256) norm_partial_kernel(const float* __restrict__ X, double* __restrict__ part,
                                                           int n, int C, int nsplit) {
  __shared__ double sh[2][8][32];
  const int b = blockIdx.y, sp = blockIdx.x;
  const int per = (n + nsplit - 1) / nsplit, tbeg = sp * per, tend = min(n, tbeg + per);
  const int cl = threadIdx.x & 31, tl = threadIdx.x >> 5;
  for (int c0 = 0; c0 < C; c0 += 32) {
    double s = 0.0, q = 0.0;
    for (int t = tbeg + tl; t < tend; t += 8) {
      const double v = (double)X[((size_t)b * n + t) * C + c0 + cl];
      s += v; q += v * v;
    }
    sh[0][tl][cl] = s; sh[1][tl][cl] = q;
    __syncthreads();
    if (tl == 0) {
      for (int i = 1; i < 8; ++i) { s += sh[0][i][cl]; q += sh[1][i][cl]; }
      double* o = part + (((size_t)b * nsplit + sp) * 2) * C;
      o[c0 + cl] = s; o[C + c0 + cl] = q;
    }
    __syncthreads();
  }
}

__global__ void norm_finish_kernel(const double* __restrict__ part, float* __restrict__ nscale, float* __restrict__ nshift,
                                   int B, int n, int C, int nsplit, int batch_mode) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * C) return;
  const int b = i / C, c = i % C;
  double s = 0.0, q = 0.0, cnt;
  if (batch_mode) {
    for (int bb = 0; bb < B; ++bb)
      for (int sp = 0; sp < nsplit; ++sp) {
        const double* o = part + (((size_t)bb * nsplit + sp) * 2) * C;
        s += o[c]; q += o[C + c];
      }
    cnt = (double)B * n;
  } else {
    for (int sp = 0; sp < nsplit; ++sp) {
      const double* o = part + (((size_t)b * nsplit + sp) * 2) * C;
      s += o[c]; q += o[C + c];
    }
    cnt = (double)n;
  }
  const double mean = s / cnt;
  double var = q / cnt - mean * mean;
  if (var < 0.0) var = 0.0;
  const double rstd = 1.0 / sqrt(var + 1e-8);
  nscale[i] = (float)rstd;
  nshift[i] = (float)(-mean * rstd);
}

int norm_stats(const Layout& L, const gf_attn_desc* d, const float* X, float* ws, cudaStream_t st) {
  if (d->norm != GF_NORM_INSTANCE && d->norm != GF_NORM_BATCH) return GF_OK;
  double* part = reinterpret_cast<double*>(ws + L.w_NPART);
  norm_partial_kernel<<<dim3(L.nsplit_norm, L.B), 256, 0, st>>>(X, part, L.n, L.C, L.nsplit_norm);
  GF_LAUNCH_OK();
  norm_finish_kernel<<<(L.B * L.C + 255) / 256, 256, 0, st>>>(part, ws + L.w_NSCALE, ws + L.w_NSHIFT, L.B, L.n, L.C,
                                                               L.nsplit_norm, d->norm == GF_NORM_BATCH ? 1 : 0);
  GF_LAUNCH_OK();
  return GF_OK;
}

// ------------------------------------------------------------------------------------------------------
// duplex pass A: latents attend to the grid.  Xbar[b,j,:] = sum_t softmax_t(L[b,t,j]) x[b,t,:]
// ------------------------------------------------------------------------------------------------------
// grid (nsplit, B): each CTA streams a contiguous token range of one image with an online softmax per latent
// and writes a partial (acc[KP][C], m[KP], l[KP]); merge kernel combines the splits deterministically.
struct CenParams {
  const float* X; const float* M; const float* Rt; const float* Ct; float* part;
  int n, H, W, C, k, nsplit;
};

template <int KP>
__global__ void __launch_bounds__(TM) centroid_simt_kernel(const CenParams P) {
  extern __shared__ __align__(16) float dyn[];            // acc [KP][C]
  __shared__ __align__(16) float xs[TM][XS];
  __shared__ __align__(16) float ks[KP][CH];
  __shared__ __align__(16) float es[TM][KP];              // logits, then exp weights
  __shared__ float red[4][KP];
  __shared__ float m_run[KP], l_run[KP], resc[KP];

  const int b = blockIdx.y, sp = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = P.n, C = P.C, k = P.k;
  const float* Xb = P.X + (size_t)b * n * C;
  const float* Mb = P.M + (size_t)b * KP * C;
  float* acc = dyn;
  const int tiles = (n + TM - 1) / TM, per = (tiles + P.nsplit - 1) / P.nsplit;
  const int tile_beg = sp * per, tile_end = min(tiles, tile_beg + per);

  for (int i = tid; i < KP * C; i += TM) acc[i] = 0.f;
  if (tid < KP) { m_run[tid] = -INFINITY; l_run[tid] = 0.f; }

  for (int tile = tile_beg; tile < tile_end; ++tile) {
    const int t0 = tile * TM, t = t0 + tid;
    const bool valid = t < n;
    float s[KP];
    {
      const int h = valid ? t / P.W : 0, w = valid ? t % P.W : 0;
      const float* rt = P.Rt + ((size_t)b * P.H + h) * KP;
      const float* ct = P.Ct + ((size_t)b * P.W + w) * KP;
#pragma unroll
      for (int j = 0; j < KP; ++j) s[j] = rt[j] + ct[j];
    }
    for (int c0 = 0; c0 < C; c0 += CH) {
      __syncthreads();
      load_x_chunk(xs, Xb, t0, n, C, c0);
      for (int i = tid; i < KP * CH / 4; i += TM) {
        const int j = i / (CH / 4), c4 = (i % (CH / 4)) * 4;
        *reinterpret_cast<float4*>(&ks[j][c4]) = __ldg(reinterpret_cast<const float4*>(Mb + (size_t)j * C + c0 + c4));
      }
      __syncthreads();
#pragma unroll
      for (int c4 = 0; c4 < CH; c4 += 4) {
        const float4 x = *reinterpret_cast<const float4*>(&xs[tid][c4]);
#pragma unroll
        for (int j = 0; j < KP; ++j) {
          const float4 kv = *reinterpret_cast<const float4*>(&ks[j][c4]);
          s[j] = fmaf(x.x, kv.x, fmaf(x.y, kv.y, fmaf(x.z, kv.z, fmaf(x.w, kv.w, s[j]))));
        }
      }
    }
    // tile maximum per latent (warp shuffle, then across the 4 warps)
#pragma unroll
    for (int j = 0; j < KP; ++j) {
      float v = valid ? s[j] : -INFINITY;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
      if (lane == 0) red[wid][j] = v;
    }
    __syncthreads();
    if (tid < KP) {
      const float tm = fmaxf(fmaxf(red[0][tid], red[1][tid]), fmaxf(red[2][tid], red[3][tid]));
      const float mo = m_run[tid], mn = fmaxf(mo, tm);
      // padded latents (j >= k) have -inf everywhere: keep them inert
      resc[tid] = (mn == -INFINITY) ? 1.f : __expf(mo - mn);
      m_run[tid] = mn;
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < KP; ++j) {
      const float mn = m_run[j];
      es[tid][j] = (valid && mn != -INFINITY) ? __expf(s[j] - mn) : 0.f;
    }
    __syncthreads();
    // running denominators
    if (tid < KP) {
      float a = 0.f;
      for (int tt = 0; tt < TM; ++tt) a += es[tt][tid];
      l_run[tid] = l_run[tid] * resc[tid] + a;
    }
    // acc[j][c] = acc[j][c]*resc[j] + sum_t e[t][j] x[t][c]; thread -> (channel lane, group of KP/4 latents)
    constexpr int JG = KP / 4;
    for (int c0 = 0; c0 < C; c0 += CH) {
      __syncthreads();
      load_x_chunk(xs, Xb, t0, n, C, c0);
      __syncthreads();
      float a[JG];
#pragma unroll
      for (int q = 0; q < JG; ++q) a[q] = 0.f;
      for (int tt = 0; tt < TM; ++tt) {
        const float x = xs[tt][lane];
#pragma unroll
        for (int q = 0; q < JG; ++q) a[q] = fmaf(es[tt][wid * JG + q], x, a[q]);
      }
#pragma unroll
      for (int q = 0; q < JG; ++q) {
        const int j = wid * JG + q;
        float* p = acc + (size_t)j * C + c0 + lane;
        *p = fmaf(*p, resc[j], a[q]);
      }
    }
    __syncthreads();
  }
  __syncthreads();
  float* out = P.part + ((size_t)b * P.nsplit + sp) * KP * (C + 4);
  for (int i = tid; i < KP * C; i += TM) out[(size_t)(i / C) * (C + 4) + (i % C)] = acc[i];
  if (tid < KP) { out[(size_t)tid * (C + 4) + C] = m_run[tid]; out[(size_t)tid * (C + 4) + C + 1] = l_run[tid]; }
  (void)k;
}

// xbar[b,j,c] = sum_sp exp(m_sp - m) acc_sp[j][c] / sum_sp exp(m_sp - m) l_sp;  lse[b,j] = m + log(sum_sp exp(m_sp - m) l_sp)
__global__ void centroid_merge_kernel(const float* __restrict__ part, float* __restrict__ xbar, int B, int k, int KP, int C, int nsplit,
                                      const float* __restrict__ in_scale, int in_ld, float* __restrict__ lse) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * k * C) return;
  const int c = i % C, j = (i / C) % k, b = i / (C * k);
  const float* base = part + (size_t)b * nsplit * KP * (C + 4) + (size_t)j * (C + 4);
  float m = -INFINITY;
  for (int sp = 0; sp < nsplit; ++sp) m = fmaxf(m, base[(size_t)sp * KP * (C + 4) + C]);
  float num = 0.f, den = 0.f;
  for (int sp = 0; sp < nsplit; ++sp) {
    const float* o = base + (size_t)sp * KP * (C + 4);
    const float ms = o[C];
    const float wgt = (ms == -INFINITY) ? 0.f : __expf(ms - m);
    num = fmaf(wgt, o[c], num);
    den = fmaf(wgt, o[C + 1], den);
  }
  xbar[i] = num / den * (in_scale ? in_scale[(size_t)b * in_ld + c] : 1.f);     // Xbar of x_in = x * d
  if (lse && c == 0) lse[(size_t)b * k + j] = m + logf(den);
}

int centroid_pass_simt(const Layout& L, const gf_attn_desc* d, const float* X, float* ws, cudaStream_t st, const float* in_scale, int in_scale_ld) {
  (void)d;
  int rc = centroid_partials_simt(L, X, ws + L.w_M, ws + L.w_Rt2, ws + L.w_Ct2, ws + L.w_PART, st);
  if (rc) return rc;
  return centroid_merge(L, ws, st, in_scale, in_scale_ld);
}

int centroid_partials_simt(const Layout& L, const float* X, const float* M, const float* Rt, const float* Ct, float* part, cudaStream_t st) {
  CenParams P;
  P.X = X; P.M = M; P.Rt = Rt; P.Ct = Ct; P.part = part;
  P.n = L.n; P.H = L.H; P.W = L.W; P.C = L.C; P.k = L.k; P.nsplit = L.nsplit_cen;
  const size_t dyn = (size_t)L.KP * L.C * sizeof(float);
  dim3 grid(L.nsplit_cen, L.B);
  if (L.KP == 16) {
    GF_CUDA_OK(cudaFuncSetAttribute(centroid_simt_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    centroid_simt_kernel<16><<<grid, TM, dyn, st>>>(P);
  } else {
    GF_CUDA_OK(cudaFuncSetAttribute(centroid_simt_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    centroid_simt_kernel<32><<<grid, TM, dyn, st>>>(P);
  }
  GF_LAUNCH_OK();
  return GF_OK;
}

int centroid_merge(const Layout& L, float* ws, cudaStream_t st, const float* in_scale, int in_scale_ld, float* xbar, float* lse) {
  const int tot = L.B * L.k * L.C;
  centroid_merge_kernel<<<(tot + 255) / 256, 256, 0, st>>>(ws + L.w_PART, xbar ? xbar : ws + L.w_XBAR, L.B, L.k, L.KP, L.C, L.nsplit_cen,
                                                           in_scale, in_scale_ld, lse);
  GF_LAUNCH_OK();
  return GF_OK;
}

}  // namespace gf
