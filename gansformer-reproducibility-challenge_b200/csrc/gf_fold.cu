// gf_fold.cu -- stage W (weight folding) and stage I (per-image prologue) of the bipartite attention block.
//
// Replaces, on the reference side (expected src/training/network.py, not in the checkout): dense_layer /
// get_weight (equalised-LR scaling), the K and V dense layers of transformer_layer, and
// get_positional_embeddings.  Buffer layouts mirror oracle/folded.py: fold_weights(), prologue().
#include <stdlib.h>
#include "gf_common.cuh"

namespace gf {

// ------------------------------------------------------------------------------------------------------
// layout
// ------------------------------------------------------------------------------------------------------
int make_layout(const gf_attn_desc* d, Layout* L) {
  if (!d) { set_error("null descriptor"); return GF_ERR_INVALID; }
  if (d->B <= 0 || d->H <= 0 || d->W <= 0 || d->C <= 0 || d->k <= 0 || d->D <= 0) {
    set_error("non-positive dimension in descriptor (B=%d H=%d W=%d C=%d k=%d D=%d)", d->B, d->H, d->W, d->C, d->k, d->D);
    return GF_ERR_INVALID;
  }
  if (d->C % 32 != 0 || d->C > 1024) { set_error("C=%d unsupported: need C %% 32 == 0 and C <= 1024", d->C); return GF_ERR_UNSUPPORTED; }
  if (d->k > 32) { set_error("k=%d unsupported: at most 32 latents", d->k); return GF_ERR_UNSUPPORTED; }
  if (d->D > 256) { set_error("D=%d unsupported: latent size at most 256", d->D); return GF_ERR_UNSUPPORTED; }
  if (d->duplex < 0 || d->duplex > 16) { set_error("duplex=%d: 0 (simplex) or the number of k-means iterations (1..16)", d->duplex); return GF_ERR_INVALID; }
  if (d->heads < 1) { set_error("num_heads=%d: must be >= 1", d->heads); return GF_ERR_INVALID; }
  if (d->heads > 1) {
    // multi-head stage T: the heads become column segments of the per-image tables (K' / V^T / Rt / Ct hold heads * seg "latents",
    // the softmax runs per segment).  Segments of 8, 16 or 32 columns; heads * seg <= 32.
    int seg = d->k <= 8 ? 8 : (d->k <= 16 ? 16 : 32);
    if (d->C % d->heads != 0 || ((d->C / d->heads) & 3)) { set_error("num_heads=%d must divide C=%d into multiples of 4 channels", d->heads, d->C); return GF_ERR_UNSUPPORTED; }
    if (d->heads != 2 && d->heads != 4) { set_error("num_heads=%d unsupported: 1, 2 or 4 heads", d->heads); return GF_ERR_UNSUPPORTED; }
    if (d->heads * seg > 32) { set_error("num_heads=%d with k=%d needs %d table columns: at most 32 (heads * k rounded up to 8 / 16)", d->heads, d->k, d->heads * seg); return GF_ERR_UNSUPPORTED; }
    if (d->duplex) { set_error("num_heads > 1 is implemented for simplex layers (duplex: 1 head)"); return GF_ERR_UNSUPPORTED; }
  }
  if (d->norm < GF_NORM_NONE || d->norm > GF_NORM_BATCH) { set_error("bad norm %d", d->norm); return GF_ERR_INVALID; }
  if (d->integration < GF_INT_MUL || d->integration > GF_INT_BOTH) { set_error("bad integration %d", d->integration); return GF_ERR_INVALID; }
  if (d->pos_dim < 0 || d->pos_dim % 4 != 0 || d->pos_dim > 256) { set_error("pos_dim=%d unsupported: need multiple of 4, <= 256", d->pos_dim); return GF_ERR_UNSUPPORTED; }
  if ((long long)d->B * d->H * d->W > (1ll << 31) - 1) { set_error("B*H*W overflows int32"); return GF_ERR_UNSUPPORTED; }

  Layout& l = *L;
  l.B = d->B; l.H = d->H; l.W = d->W; l.C = d->C; l.k = d->k; l.D = d->D; l.p = d->pos_dim;
  l.heads = d->heads;
  l.seg = d->heads > 1 ? (d->k <= 8 ? 8 : (d->k <= 16 ? 16 : 32)) : pad_k(d->k);
  l.KP = d->heads > 1 ? pad_k(l.heads * l.seg) : pad_k(d->k);
  // heads in {2, 4} and seg in {8, 16}: heads * seg is 16 or 32, i.e. KP == heads * seg
  l.Cout = d->integration == GF_INT_BOTH ? 2 * d->C : d->C;
  l.LDK = (d->C + d->pos_dim + 4 + 3) & ~3;          // rows of the [.., LDK] matrices are read as float4
  l.n = d->H * d->W;
  l.duplex = d->duplex ? 1 : 0;
  const size_t C = l.C, k = l.k, D = l.D, p = l.p, LDK = l.LDK;
  const size_t Din = l.duplex ? C : D;

  size_t o = 0;
  auto take = [&](size_t nfloats) { size_t r = o; o += align64(nfloats); return r; };
  const size_t nh = l.heads;                         // per-head copies of the key / value folds (simplex)
  l.f_AK = take(nh * Din * LDK);
  l.f_CK = take(nh * k * LDK);
  l.f_AV = take(nh * D * l.Cout);
  l.f_CV = take(nh * l.Cout);
  l.f_CB = take(l.Cout);
  l.f_ROW = take((size_t)l.H * (p / 2) + 1);
  l.f_COL = take((size_t)l.W * (p / 2) + 1);
  l.f_QFOLD = take(C * LDK);
  l.f_KCONST = take(k * C);
  if (l.duplex) {
    l.f_WV2 = take(C * C);
    l.f_BV2 = take(C);
    l.f_AK2 = take(C * LDK);
    l.f_CK2 = take(k * LDK);
    l.f_AM = take(D * LDK);
    l.f_CM = take(k * LDK);
    l.f_MFOLD = take(C * LDK);
    l.f_QCONST = take(k * C);
    l.f_ACQ = (d->duplex > 1 || (d->flags & GF_FLAG_CENTROIDS_INIT)) ? take(C * LDK) : 0;
    l.f_WI2L = (d->flags & GF_FLAG_IMG2LTNT) ? take(C * D) : 0;
    l.f_BI2L = (d->flags & GF_FLAG_IMG2LTNT) ? take(D) : 0;
  } else {
    l.f_WV2 = l.f_BV2 = l.f_AM = l.f_CM = l.f_MFOLD = l.f_QCONST = l.f_AK2 = l.f_CK2 = l.f_ACQ = l.f_WI2L = l.f_BI2L = 0;
  }
  l.iters = d->duplex;
  l.img2ltnt = (d->duplex && (d->flags & GF_FLAG_IMG2LTNT)) ? 1 : 0;
  l.f_total = o;

  // statistics / centroid splits: about two waves of CTAs over the device's SMs
  const int sms = num_sms();
  int want = (2 * sms + l.B - 1) / l.B;
  l.nsplit_norm = want; if (l.nsplit_norm > (l.n + 63) / 64) l.nsplit_norm = (l.n + 63) / 64; if (l.nsplit_norm < 1) l.nsplit_norm = 1;
  {
    // centroid splits: one CTA per SM.  Cost model in tile units: every CTA pays a fixed cost (TMEM allocation, loading M,
    // flushing its [KP, C] partial -- about two tiles' worth) plus its share of the image's tiles, and the grid runs in
    // ceil(CTAs / SMs) rounds.  Small images therefore get ONE split (a 32x32 grid used to be cut into 8 one-tile CTAs, each
    // moving as many bytes of M and partials as of X).
    const int tiles = (l.n + 127) / 128;
    const int z = l.C == 512 ? 2 : 1;                   // C = 512: two CTAs per split (channel halves)
    int best = 1;
    long long best_cost = -1;
    for (int ns = 1; ns <= 16 && ns <= tiles; ++ns) {
      const long long rounds = ((long long)l.B * ns * z + sms - 1) / sms;
      const long long cost = rounds * ((tiles + ns - 1) / ns + 2);
      if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = ns; }
    }
    l.nsplit_cen = best;
    static const int forced = []() { const char* e = getenv("GF_NSPLIT_CEN"); return e ? atoi(e) : 0; }();   // tuning aid, read once per process
    if (forced >= 1 && forced <= 16 && forced <= tiles) l.nsplit_cen = forced;
  }

  o = 0;
  const size_t B = l.B, KP = l.KP;
  l.w_KPALL = take(B * k * LDK);
  l.w_Kp = take(B * KP * C);
  l.w_Vt = take(B * l.Cout * KP);
  l.w_Rt = take(B * l.H * KP);
  l.w_Ct = take(B * l.W * KP);
  l.w_CB = take(l.Cout);
  if (d->norm == GF_NORM_INSTANCE || d->norm == GF_NORM_BATCH) {
    l.w_NSCALE = take(B * C);
    l.w_NSHIFT = take(B * C);
    l.w_NPART = take(B * (size_t)l.nsplit_norm * 2 * C * 2);  // doubles
  } else {
    l.w_NSCALE = l.w_NSHIFT = l.w_NPART = 0;
  }
  if (l.duplex) {
    l.w_MALL = take(B * k * LDK);
    l.w_M = take(B * KP * C);
    l.w_Rt2 = take(B * l.H * KP);
    l.w_Ct2 = take(B * l.W * KP);
    l.w_PART = take(B * (size_t)l.nsplit_cen * KP * (C + 4));
    l.w_XBAR = take(B * k * C);
    l.w_CEN = take(B * k * C);
    l.w_Y2 = take(B * k * D);
  } else {
    l.w_MALL = l.w_M = l.w_Rt2 = l.w_Ct2 = l.w_PART = l.w_XBAR = l.w_CEN = l.w_Y2 = 0;
  }
  l.w_total = o;
  return GF_OK;
}

// ------------------------------------------------------------------------------------------------------
// small SGEMM used by the folding stages (weights-only / per-image [B*k] rows: tiny problems)
// ------------------------------------------------------------------------------------------------------
template <bool TA, bool TB>
__global__ void __launch_bounds__(256) gemm_kernel(int M, int N, int K, const float* __restrict__ A, int lda,
                                                   const float* __restrict__ Bm, int ldb, float* __restrict__ Cm, int ldc,
                                                   float alpha, const float* __restrict__ E, int lde, int emod,
                                                   const float* __restrict__ v) {
  __shared__ float As[32][33];
  __shared__ float Bs[32][33];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int m0 = blockIdx.y * 32, n0 = blockIdx.x * 32;
  float acc[2][2] = {{0.f, 0.f}, {0.f, 0.f}};
  for (int k0 = 0; k0 < K; k0 += 32) {
    for (int i = threadIdx.x; i < 1024; i += 256) {
      const int r = i >> 5, c = i & 31;
      const int m = m0 + r, kk = k0 + c;
      As[r][c] = (m < M && kk < K) ? (TA ? A[(size_t)kk * lda + m] : A[(size_t)m * lda + kk]) : 0.f;
      const int kb = k0 + r, nn = n0 + c;
      Bs[r][c] = (kb < K && nn < N) ? (TB ? Bm[(size_t)nn * ldb + kb] : Bm[(size_t)kb * ldb + nn]) : 0.f;
    }
    __syncthreads();
#pragma unroll 8
    for (int kk = 0; kk < 32; ++kk) {
      const float a0 = As[ty * 2][kk], a1 = As[ty * 2 + 1][kk];
      const float b0 = Bs[kk][tx * 2], b1 = Bs[kk][tx * 2 + 1];
      acc[0][0] = fmaf(a0, b0, acc[0][0]); acc[0][1] = fmaf(a0, b1, acc[0][1]);
      acc[1][0] = fmaf(a1, b0, acc[1][0]); acc[1][1] = fmaf(a1, b1, acc[1][1]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int m = m0 + ty * 2 + i, nn = n0 + tx * 2 + j;
      if (m < M && nn < N) {
        float r = alpha * acc[i][j];
        if (E) r += E[(size_t)(m % emod) * lde + nn];
        if (v) r += v[nn];
        Cm[(size_t)m * ldc + nn] = r;
      }
    }
}

// Register-blocked NN SGEMM for the per-image [B*k, C] x [C, C(+p+4)] products of the duplex path: 64x64 block tile,
// BK = 16, 256 threads x (4x4) outputs, float4 shared-memory reads.  Requires lda, ldb % 4 == 0 and 16-byte aligned bases.
__global__ void __launch_bounds__(256) gemm64_kernel(int M, int N, int K, const float* __restrict__ A, int lda,
                                                     const float* __restrict__ Bm, int ldb, float* __restrict__ Cm, int ldc,
                                                     float alpha, const float* __restrict__ E, int lde, int emod,
                                                     const float* __restrict__ v) {
  __shared__ __align__(16) float As[16][64 + 4];     // [k][m] (transposed on load)
  __shared__ __align__(16) float Bs[16][64 + 4];     // [k][n]
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  const int ar = tid >> 2, ac = (tid & 3) * 4;       // A tile 64 x 16: row ar, cols ac..ac+3
  const int br = tid >> 4, bc = (tid & 15) * 4;      // B tile 16 x 64: row br, cols bc..bc+3
  for (int k0 = 0; k0 < K; k0 += 16) {
    float4 a4 = make_float4(0.f, 0.f, 0.f, 0.f), b4 = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m0 + ar < M) {
      if (k0 + ac + 3 < K) a4 = *reinterpret_cast<const float4*>(A + (size_t)(m0 + ar) * lda + k0 + ac);
      else {
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = 0; i < 4; ++i) if (k0 + ac + i < K) t[i] = A[(size_t)(m0 + ar) * lda + k0 + ac + i];
        a4 = make_float4(t[0], t[1], t[2], t[3]);
      }
    }
    if (k0 + br < K) {
      if (n0 + bc + 3 < N) b4 = *reinterpret_cast<const float4*>(Bm + (size_t)(k0 + br) * ldb + n0 + bc);
      else {
        float t[4] = {0.f, 0.f, 0.f, 0.f};
        for (int i = 0; i < 4; ++i) if (n0 + bc + i < N) t[i] = Bm[(size_t)(k0 + br) * ldb + n0 + bc + i];
        b4 = make_float4(t[0], t[1], t[2], t[3]);
      }
    }
    __syncthreads();
    As[ac + 0][ar] = a4.x; As[ac + 1][ar] = a4.y; As[ac + 2][ar] = a4.z; As[ac + 3][ar] = a4.w;
    *reinterpret_cast<float4*>(&Bs[br][bc]) = b4;
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int nn = n0 + tx * 4 + j;
      if (nn >= N) continue;
      float r = alpha * acc[i][j];
      if (E) r += E[(size_t)(m % emod) * lde + nn];
      if (v) r += v[nn];
      Cm[(size_t)m * ldc + nn] = r;
    }
  }
}

int gemm(cudaStream_t st, int M, int N, int K, const float* A, int lda, bool ta, const float* B, int ldb, bool tb,
         float* Cm, int ldc, float alpha, const float* E, int lde, int emod, const float* v, bool allow_tf32) {
  if (M <= 0 || N <= 0) return GF_OK;
  if (allow_tf32 && !ta && !tb && lda == K && ldb == N && gemm_tc_ok(M, N, K, A, B, Cm, ldc))
    return gemm_tc(st, M, N, K, A, B, Cm, ldc, alpha, E, lde, emod, v);
  if (!ta && !tb && M >= 256 && N >= 64 && K >= 64 && (lda & 3) == 0 && (ldb & 3) == 0 && ((uintptr_t)A & 15) == 0 && ((uintptr_t)B & 15) == 0) {
    if (emod < 1) emod = 1;
    gemm64_kernel<<<dim3((N + 63) / 64, (M + 63) / 64), 256, 0, st>>>(M, N, K, A, lda, B, ldb, Cm, ldc, alpha, E, lde, emod, v);
    GF_LAUNCH_OK();
    return GF_OK;
  }
  dim3 grid((N + 31) / 32, (M + 31) / 32);
  if (emod < 1) emod = 1;
  if (!ta && !tb) gemm_kernel<false, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, Cm, ldc, alpha, E, lde, emod, v);
  else if (ta && !tb) gemm_kernel<true, false><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, Cm, ldc, alpha, E, lde, emod, v);
  else if (!ta && tb) gemm_kernel<false, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, Cm, ldc, alpha, E, lde, emod, v);
  else gemm_kernel<true, true><<<grid, 256, 0, st>>>(M, N, K, A, lda, B, ldb, Cm, ldc, alpha, E, lde, emod, v);
  GF_LAUNCH_OK();
  return GF_OK;
}

// ------------------------------------------------------------------------------------------------------
// stage W helper kernels
// ------------------------------------------------------------------------------------------------------
// out[c', col], c' < C, col < LDK:  [ Wq^T * a | Wp^T * ap | bias * s | 0 0 0 ]   (oracle/folded.py: qfold / m_fold)
__global__ void build_fold_kernel(float* __restrict__ out, const float* __restrict__ wq, const float* __restrict__ wp,
                                  const float* __restrict__ bias, int C, int p, int LDK, float a, float ap, float s) {
  const size_t total = (size_t)C * LDK;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int cp = (int)(i / LDK), col = (int)(i % LDK);
    float r = 0.f;
    if (col < C) r = wq[(size_t)col * C + cp] * a;
    else if (col < C + p) r = wp ? wp[(size_t)(col - C) * C + cp] * ap : 0.f;
    else if (col == C + p) r = bias ? bias[cp] * s : 0.f;
    out[i] = r;
  }
}

__global__ void scale_copy_kernel(float* __restrict__ out, const float* __restrict__ in, size_t nel, float a, float add, size_t add_upto) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < nel; i += (size_t)gridDim.x * blockDim.x)
    out[i] = in[i] * a + (i < add_upto ? add : 0.f);
}

// sinusoidal_axis(length, dim): [sin(pos*f_m) m<dim/2 | cos(pos*f_m)], f_m = (pi/2) 2^m, pos = (i+.5)/length*2-1
__global__ void pos_axis_kernel(float* __restrict__ out, int length, int dim) {
  const int total = length * dim;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int r = i / dim, q = i % dim, hq = dim / 2;
    const double pos = ((double)r + 0.5) / (double)length * 2.0 - 1.0;
    const int m = q < hq ? q : q - hq;
    const double ang = pos * (1.5707963267948966 * exp2((double)m));
    out[i] = (float)(q < hq ? sin(ang) : cos(ang));
  }
}

// out[j, :] = row0(out) + add[j, :] for j = k-1 .. 0 (row 0 last: it is the source)
__global__ void bias_rows_kernel(float* __restrict__ out, const float* __restrict__ add, int k, int ld) {
  for (size_t c = blockIdx.x * (size_t)blockDim.x + threadIdx.x; c < (size_t)ld; c += (size_t)gridDim.x * blockDim.x) {
    const float r0 = out[c];
    for (int j = k - 1; j >= 0; --j) out[(size_t)j * ld + c] = r0 + add[(size_t)j * ld + c];
  }
}

static inline int blocks_for(size_t nel) { size_t b = (nel + 255) / 256; return (int)(b > 1184 ? 1184 : (b < 1 ? 1 : b)); }

int fold_weights(const Layout& L, const gf_attn_desc* d, const gf_attn_weights* w, float* f, cudaStream_t st) {
  const int C = L.C, k = L.k, D = L.D, p = L.p, LDK = L.LDK, Cout = L.Cout;
  const bool pos = p > 0;
  if (!w->wq || !w->bq || !w->bk || !w->wv || !w->bv || !w->wo || !w->bo) { set_error("fold_weights: null simplex weight pointer"); return GF_ERR_INVALID; }
  if (pos && (!w->wpq || !w->wpk || !w->pos_latent)) { set_error("fold_weights: pos_dim>0 but positional weights are null"); return GF_ERR_INVALID; }
  if (!L.duplex && !w->wk) { set_error("fold_weights: null wk"); return GF_ERR_INVALID; }
  if (L.duplex && (!w->wq2 || !w->bq2 || !w->wk2 || !w->wv2 || !w->bv2 || !w->wkc || (pos && (!w->wpq2 || !w->wpk2)))) {
    set_error("fold_weights: duplex weights are null"); return GF_ERR_INVALID;
  }
  const int nh = L.heads, ch = C / nh;            // channels per head
  const float s = 1.f / sqrtf((float)ch);         // 1/sqrt(C/heads)
  const float rC = 1.f / sqrtf((float)C), rD = 1.f / sqrtf((float)D), rp = pos ? 1.f / sqrtf((float)p) : 0.f;
  int rc;
  // qfold [C, LDK]
  build_fold_kernel<<<blocks_for((size_t)C * LDK), 256, 0, st>>>(f + L.f_QFOLD, w->wq, pos ? w->wpq : nullptr, w->bq, C, p, LDK, s * rC, s * rp, s);
  GF_LAUNCH_OK();
  // kconst [k, C] = bk + Pl @ wpk_e
  if ((rc = gemm(st, k, C, pos ? p : 0, w->pos_latent, p, false, w->wpk, C, false, f + L.f_KCONST, C, rp, nullptr, 0, 1, w->bk))) return rc;
  // CK = kconst @ qfold
  if ((rc = gemm(st, k, LDK, C, f + L.f_KCONST, C, false, f + L.f_QFOLD, LDK, false, f + L.f_CK, LDK, 1.f))) return rc;
  if (L.duplex) {
    // AK [C, LDK] = wkc_e @ qfold  (applied to centroids)
    if ((rc = gemm(st, C, LDK, C, w->wkc, C, false, f + L.f_QFOLD, LDK, false, f + L.f_AK, LDK, rC))) return rc;
    scale_copy_kernel<<<blocks_for((size_t)C * C), 256, 0, st>>>(f + L.f_WV2, w->wv2, (size_t)C * C, rC, 0.f, 0);
    GF_LAUNCH_OK();
    scale_copy_kernel<<<blocks_for(C), 256, 0, st>>>(f + L.f_BV2, w->bv2, C, 1.f, 0.f, 0);
    GF_LAUNCH_OK();
    // keys straight from Xbar when the caller does not ask for the centroids: (Xbar Wv2 + bv2) AK + CK = Xbar AK2 + CK2
    if ((rc = gemm(st, C, LDK, C, f + L.f_WV2, C, false, f + L.f_AK, LDK, false, f + L.f_AK2, LDK, 1.f))) return rc;
    if ((rc = gemm(st, 1, LDK, C, f + L.f_BV2, C, false, f + L.f_AK, LDK, false, f + L.f_CK2, LDK, 1.f))) return rc;      // row 0 = bv2 AK
    bias_rows_kernel<<<blocks_for((size_t)k * LDK), 256, 0, st>>>(f + L.f_CK2, f + L.f_CK, k, LDK);
    GF_LAUNCH_OK();
    // pass A: mfold [C, LDK] (no bias column: the bk2 term is constant over n and cancels in softmax_n)
    build_fold_kernel<<<blocks_for((size_t)C * LDK), 256, 0, st>>>(f + L.f_MFOLD, w->wk2, pos ? w->wpk2 : nullptr, nullptr, C, p, LDK, s * rC, s * rp, 0.f);
    GF_LAUNCH_OK();
    if ((rc = gemm(st, k, C, pos ? p : 0, w->pos_latent, p, false, w->wpq2, C, false, f + L.f_QCONST, C, rp, nullptr, 0, 1, w->bq2))) return rc;
    if ((rc = gemm(st, D, LDK, C, w->wq2, C, false, f + L.f_MFOLD, LDK, false, f + L.f_AM, LDK, rD))) return rc;
    if ((rc = gemm(st, k, LDK, C, f + L.f_QCONST, C, false, f + L.f_MFOLD, LDK, false, f + L.f_CM, LDK, 1.f))) return rc;
    if (L.f_ACQ) {              // k-means iterations >= 2 / carried-in centroids: queries from the centroids, M = Cen (wcq_e mfold) + CM
      if (!w->wcq) { set_error("fold_weights: desc.duplex > 1 / GF_FLAG_CENTROIDS_INIT need wcq"); return GF_ERR_INVALID; }
      if ((rc = gemm(st, C, LDK, C, w->wcq, C, false, f + L.f_MFOLD, LDK, false, f + L.f_ACQ, LDK, rC))) return rc;
    }
    if (L.img2ltnt) {
      if (!w->wi2l || !w->bi2l) { set_error("fold_weights: GF_FLAG_IMG2LTNT needs wi2l and bi2l"); return GF_ERR_INVALID; }
      scale_copy_kernel<<<blocks_for((size_t)C * D), 256, 0, st>>>(f + L.f_WI2L, w->wi2l, (size_t)C * D, rC, 0.f, 0);
      GF_LAUNCH_OK();
      scale_copy_kernel<<<blocks_for(D), 256, 0, st>>>(f + L.f_BI2L, w->bi2l, D, 1.f, 0.f, 0);
      GF_LAUNCH_OK();
    }
  } else {
    // per head h: the key's channels of that head only -- AK_h = wk_e[:, h] qfold[h, :],  CK_h = kconst[:, h] qfold[h, :]
    for (int h = 0; h < nh; ++h) {
      if ((rc = gemm(st, D, LDK, ch, w->wk + h * ch, C, false, f + L.f_QFOLD + (size_t)h * ch * LDK, LDK, false,
                     f + L.f_AK + (size_t)h * D * LDK, LDK, rD)))
        return rc;
      if (h > 0 && (rc = gemm(st, k, LDK, ch, f + L.f_KCONST + h * ch, C, false, f + L.f_QFOLD + (size_t)h * ch * LDK, LDK, false,
                              f + L.f_CK + (size_t)h * k * LDK, LDK, 1.f)))
        return rc;
    }
    if (nh > 1 && (rc = gemm(st, k, LDK, ch, f + L.f_KCONST, C, false, f + L.f_QFOLD, LDK, false, f + L.f_CK, LDK, 1.f))) return rc;   // head 0 (overwrites the full-C product)
  }
  // per head: AV_h [D, Cout] = wv_e[:, h] @ wo_e[h, :] ; CV_h = bv[h] @ wo_e[h, :]; head 0 also carries bo (+1 on the gain half):
  // every head's probabilities sum to one, so a constant may ride on any single head
  for (int h = 0; h < nh; ++h) {
    if ((rc = gemm(st, D, Cout, ch, w->wv + h * ch, C, false, w->wo + (size_t)h * ch * Cout, Cout, false, f + L.f_AV + (size_t)h * D * Cout, Cout, rD * rC))) return rc;
    if ((rc = gemm(st, 1, Cout, ch, w->bv + h * ch, C, false, w->wo + (size_t)h * ch * Cout, Cout, false, f + L.f_CV + (size_t)h * Cout, Cout, rC,
                   nullptr, 0, 1, h == 0 ? w->bo : nullptr)))
      return rc;
  }
  if (d->integration != GF_INT_ADD) {
    scale_copy_kernel<<<blocks_for(Cout), 256, 0, st>>>(f + L.f_CV, f + L.f_CV, Cout, 1.f, 1.f, (size_t)C);
    GF_LAUNCH_OK();
  }
  // CB = bo (+1 on the gain half): with attention dropout the probabilities no longer sum to one, so the constants folded into V^T
  // are re-added as (1 - sum q) * CB by the kernels that apply the mask
  scale_copy_kernel<<<blocks_for(Cout), 256, 0, st>>>(f + L.f_CB, w->bo, Cout, 1.f, d->integration != GF_INT_ADD ? 1.f : 0.f, (size_t)C);
  GF_LAUNCH_OK();
  if (pos) {
    pos_axis_kernel<<<blocks_for((size_t)L.H * (p / 2)), 256, 0, st>>>(f + L.f_ROW, L.H, p / 2);
    GF_LAUNCH_OK();
    pos_axis_kernel<<<blocks_for((size_t)L.W * (p / 2)), 256, 0, st>>>(f + L.f_COL, L.W, p / 2);
    GF_LAUNCH_OK();
  }
  return GF_OK;
}

// ------------------------------------------------------------------------------------------------------
// stage I: per-image tables
// ------------------------------------------------------------------------------------------------------
// grid (npos + nblk, B).  blockIdx.x < npos: positional logit tables Rt/Ct of image b.  Others: Kp and (optionally) Vt.
// fp32 -> nearest-even TF32 (10 mantissa bits).  The tensor cores TRUNCATE fp32 operands to TF32; pre-rounding the
// small operands (K', V^T, and P in the kernel) makes that truncation a no-op for them and halves their error.
__device__ __forceinline__ float round_tf32(float v) {
  uint32_t b = __float_as_uint(v);
  if ((b & 0x7f800000u) == 0x7f800000u) return v;      // inf / nan untouched
  b = (b + 0xFFFu + ((b >> 13) & 1u)) & 0xFFFFE000u;
  return __uint_as_float(b);
}
// Truncation of X toward zero biases every product x*K' by E[eps] = 2^-11 / ln 2 * (1/2) = 0.7213 * 2^-11 (log-uniform
// mantissa); K' is scaled up by that factor so the logits are unbiased.
#define GF_TF32_TRUNC_COMP 1.000352220f
#define GF_LOG2E 1.4426950408889634f

__global__ void __launch_bounds__(256, 4) finalize_kernel(const float* __restrict__ kpall, const float* __restrict__ Y,
                                                       const float* __restrict__ AV, const float* __restrict__ CV,
                                                       const float* __restrict__ ROW, const float* __restrict__ COL,
                                                       float* __restrict__ Kp, float* __restrict__ Vt,
                                                       float* __restrict__ Rt, float* __restrict__ Ct,
                                                       int H, int W, int C, int k, int D, int p, int KP, int Cout, int LDK,
                                                       int tf32, int npos, const float* __restrict__ in_scale, int in_ld,
                                                       const float* __restrict__ CB, float* __restrict__ CBout) {
  // grid (B, blocks): the role index is the slow grid dimension so that the longest-running role (V^T) is dispatched first
  const int b = blockIdx.x;
  const float* kp = kpall + (size_t)b * k * LDK;
  const int nvblk = Vt ? (Cout + 255) / 256 : 0;                 // V^T role: one thread per channel
  const int blk = blockIdx.y;
  if (blk < nvblk) {
    // V^T[b, c, :] = (Y[b] . AV[:, c] + CV[c]) for the k latents (zero for the padded ones); AV reads coalesced over c
    extern __shared__ float ysm[];                                // Y[b]: k x D
    for (int i = threadIdx.x; i < k * D; i += blockDim.x) ysm[i] = Y[(size_t)b * k * D + i];
    __syncthreads();
    const int c = blk * 256 + threadIdx.x;
    if (c >= Cout) return;
    // 16 latents at a time: keeps the whole kernel at <= 64 registers (every role shares one register allocation, and at 144
    // registers only ONE 256-thread CTA fitted an SM: the ~700 latency-bound CTAs of a launch ran in five rounds)
    const float cv = CV[c];
    float* out = Vt + ((size_t)b * Cout + c) * KP;
    for (int j0 = 0; j0 < KP; j0 += 16) {
      float acc[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) acc[j] = 0.f;
      for (int d0 = 0; d0 < D; d0 += 16) {
        float a[16];                                              // 16 independent loads in flight per batch
#pragma unroll
        for (int dd = 0; dd < 16; ++dd) a[dd] = d0 + dd < D ? AV[(size_t)(d0 + dd) * Cout + c] : 0.f;
#pragma unroll
        for (int dd = 0; dd < 16; ++dd) {
          if (d0 + dd < D) {
            const float* yr = ysm + (size_t)j0 * D + d0 + dd;
#pragma unroll
            for (int j = 0; j < 16; ++j) if (j0 + j < k) acc[j] = fmaf(yr[j * D], a[dd], acc[j]);
          }
        }
      }
#pragma unroll
      for (int j4 = 0; j4 < 4; ++j4) {
        float4 r;
        r.x = j0 + j4 * 4 + 0 < k ? acc[j4 * 4 + 0] + cv : 0.f; r.y = j0 + j4 * 4 + 1 < k ? acc[j4 * 4 + 1] + cv : 0.f;
        r.z = j0 + j4 * 4 + 2 < k ? acc[j4 * 4 + 2] + cv : 0.f; r.w = j0 + j4 * 4 + 3 < k ? acc[j4 * 4 + 3] + cv : 0.f;
        if (tf32) { r.x = round_tf32(r.x); r.y = round_tf32(r.y); r.z = round_tf32(r.z); r.w = round_tf32(r.w); }
        reinterpret_cast<float4*>(out)[j0 / 4 + j4] = r;          // KP is 16 or 32: rows are 16-byte aligned
      }
    }
    return;
  }
  if (blk < nvblk + npos) {
    // batch-independent constant of the control signal, read by stage T when attention dropout is on (duplex layers)
    if (b == 0 && CBout)
      for (int i = (blk - nvblk) * blockDim.x + threadIdx.x; i < Cout; i += npos * blockDim.x) CBout[i] = CB[i];
    const int half = p / 2;
    for (int i = (blk - nvblk) * blockDim.x + threadIdx.x; i < (H + W) * KP; i += npos * blockDim.x) {
      const int r = i / KP, j = i % KP;
      const bool is_row = r < H;
      float val;
      if (j >= k) {
        val = is_row ? -INFINITY : 0.f;
      } else {
        const float* kj = kp + (size_t)j * LDK + C;
        float acc = 0.f;
        if (is_row) {
#pragma unroll 8
          for (int q = 0; q < half; ++q) acc = fmaf(ROW[r * half + q], kj[q], acc);
          acc += kj[p];
        } else {
#pragma unroll 8
          for (int q = 0; q < half; ++q) acc = fmaf(COL[(r - H) * half + q], kj[half + q], acc);
        }
        val = tf32 ? acc * GF_LOG2E : acc;           // tensor-path kernels take their logits in log2 units (one ex2 per latent)
      }
      if (is_row) Rt[((size_t)b * H + r) * KP + j] = val;
      else Ct[((size_t)b * W + (r - H)) * KP + j] = val;
    }
    return;
  }
  // K' role: float4 elements, four independent loads in flight per thread (one L2 round trip per batch instead of per element)
  const int C4 = C >> 2, nK4 = KP * C4;
  const int stride = (gridDim.y - npos - nvblk) * blockDim.x;
  const float4* isc4 = in_scale ? reinterpret_cast<const float4*>(in_scale + (size_t)b * in_ld) : nullptr;
  float4* Kp4 = reinterpret_cast<float4*>(Kp + (size_t)b * KP * C);
  for (int i0 = (blk - nvblk - npos) * blockDim.x + threadIdx.x; i0 < nK4; i0 += 4 * stride) {
    float4 v[4], d[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * stride;
      const int j = i / C4, c4 = i - j * C4;
      v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      d[u] = make_float4(1.f, 1.f, 1.f, 1.f);
      if (i < nK4 && j < k) {
        v[u] = *reinterpret_cast<const float4*>(kp + (size_t)j * LDK + c4 * 4);
        if (isc4) d[u] = isc4[c4];
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * stride;
      if (i < nK4) {
        float4 r = make_float4(v[u].x * d[u].x, v[u].y * d[u].y, v[u].z * d[u].z, v[u].w * d[u].w);   // x_in = x * in_scale: (x*d).K' == x.(K'*d)
        if (tf32) {
          constexpr float kf = GF_TF32_TRUNC_COMP * GF_LOG2E;
          r.x = round_tf32(r.x * kf); r.y = round_tf32(r.y * kf); r.z = round_tf32(r.z * kf); r.w = round_tf32(r.w * kf);
        }
        Kp4[i] = r;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------
// stage I in ONE launch for everything that depends on the latents only (the K = D product, the TF32 rounding, the
// positional-logit tables and V^T): replaces gemm_kernel + finalize_kernel for the simplex keys and for the duplex pass-A
// query tables.  Up to STAGE_I_MAX_JOBS layers per launch (the generator batches every layer's prologue of a step into
// one launch: they all read the same latents).  Arithmetic and operation order are those of gemm_kernel + finalize_kernel
// (fp32 FMA chain over d ascending, + constant row, * in_scale, * kf, round), so both routes produce the same bits.
// ------------------------------------------------------------------------------------------------------
constexpr int STAGE_I_MAX_JOBS = 16;
struct StageIJob {
  const float *Y, *A, *Cst, *AV, *CV, *ROW, *COL, *in_scale, *CB;
  float *Kp, *Vt, *Rt, *Ct, *CBout;
  int H, W, C, k, D, p, KP, Cout, LDK, in_ld;
  int heads, seg;                // multi-head: table column J = head * seg + j; A / Cst / AV / CV hold one copy per head
  int tf32_k, tf32_v;            // round K' (and take the logits in log2 units) / round V^T for the tcgen05 kernels
  int nvblk, npos, nkblk;        // CTAs per image and role
  int blk_begin;                 // first blockIdx.y of this job
};
struct StageIBatch { StageIJob job[STAGE_I_MAX_JOBS]; int njobs; };

__global__ void __launch_bounds__(256, 4) stage_i_kernel(const __grid_constant__ StageIBatch batch) {
  int ji = 0;
#pragma unroll 1
  while (ji + 1 < batch.njobs && (int)blockIdx.y >= batch.job[ji + 1].blk_begin) ++ji;
  const StageIJob& J = batch.job[ji];
  const int b = blockIdx.x, blk = (int)blockIdx.y - J.blk_begin;
  const int k = J.k, D = J.D, C = J.C, KP = J.KP, LDK = J.LDK, p = J.p;
  extern __shared__ float ysm[];                                  // Y[b]: k x D, then kap: k x (p + 1)
  for (int i = threadIdx.x; i < k * D; i += blockDim.x) ysm[i] = J.Y[(size_t)b * k * D + i];
  __syncthreads();
  if (blk < J.nvblk) {
    // ---- V^T[b, c, :] = Y[b] . AV[:, c] + CV[c]  (zero for the padded latents); one thread per channel
    const int Cout = J.Cout;
    const int c = blk * 256 + threadIdx.x;
    if (c >= Cout) return;
    if (b == 0 && J.CBout) J.CBout[c] = J.CB[c];                     // batch-independent constant of the control signal (dropout path)
    float* out = J.Vt + ((size_t)b * Cout + c) * KP;
    for (int j0 = 0; j0 < KP; j0 += 8) {                          // 8 table columns at a time: one head (seg >= 8)
      const int head = j0 / J.seg, jb = j0 - head * J.seg;        // latent index of column j0 inside its head
      const float* AVh = J.AV + (size_t)head * D * Cout;
      const float cv = J.CV[(size_t)head * Cout + c];
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
      for (int d0 = 0; d0 < D; d0 += 16) {
        float a[16];
#pragma unroll
        for (int dd = 0; dd < 16; ++dd) a[dd] = d0 + dd < D ? AVh[(size_t)(d0 + dd) * Cout + c] : 0.f;
#pragma unroll
        for (int dd = 0; dd < 16; ++dd) {
          if (d0 + dd < D) {
            const float* yr = ysm + (size_t)jb * D + d0 + dd;
#pragma unroll
            for (int j = 0; j < 8; ++j) if (jb + j < k) acc[j] = fmaf(yr[j * D], a[dd], acc[j]);
          }
        }
      }
#pragma unroll
      for (int j4 = 0; j4 < 2; ++j4) {
        float4 r;
        r.x = jb + j4 * 4 + 0 < k ? acc[j4 * 4 + 0] + cv : 0.f; r.y = jb + j4 * 4 + 1 < k ? acc[j4 * 4 + 1] + cv : 0.f;
        r.z = jb + j4 * 4 + 2 < k ? acc[j4 * 4 + 2] + cv : 0.f; r.w = jb + j4 * 4 + 3 < k ? acc[j4 * 4 + 3] + cv : 0.f;
        if (J.tf32_v) { r.x = round_tf32(r.x); r.y = round_tf32(r.y); r.z = round_tf32(r.z); r.w = round_tf32(r.w); }
        reinterpret_cast<float4*>(out)[j0 / 4 + j4] = r;
      }
    }
    return;
  }
  if (blk < J.nvblk + J.npos) {
    // ---- positional logit tables: kap[j, q] = (Y[b] . A + Cst)[j, C + q], q <= p (the last one is the bias column)
    float* kap = ysm + k * D;
    const int pw = p + 1;
    for (int i = threadIdx.x; i < KP * pw; i += blockDim.x) {
      const int Jc = i / pw, q = i - Jc * pw;
      const int head = Jc / J.seg, j = Jc - head * J.seg;
      if (j >= k) { kap[i] = 0.f; continue; }
      const float* Ah = J.A + (size_t)head * D * LDK;
      float acc = 0.f;
      for (int d0 = 0; d0 < D; d0 += 8) {                 // 8 independent loads in flight (one L2 round trip per batch)
        float a[8];
#pragma unroll
        for (int dd = 0; dd < 8; ++dd) a[dd] = d0 + dd < D ? Ah[(size_t)(d0 + dd) * LDK + C + q] : 0.f;
#pragma unroll
        for (int dd = 0; dd < 8; ++dd) if (d0 + dd < D) acc = fmaf(ysm[j * D + d0 + dd], a[dd], acc);
      }
      kap[i] = acc + J.Cst[((size_t)head * k + j) * LDK + C + q];
    }
    __syncthreads();
    const int half = p / 2, H = J.H, W = J.W;
    for (int i = (blk - J.nvblk) * blockDim.x + threadIdx.x; i < (H + W) * KP; i += J.npos * blockDim.x) {
      const int r = i / KP, j = i % KP;
      const bool is_row = r < H;
      float val;
      if (j % J.seg >= k) {                          // padded column of its head: probability exactly 0
        val = is_row ? -INFINITY : 0.f;
      } else {
        const float* kj = kap + j * pw;
        float acc = 0.f;
        if (is_row) {
#pragma unroll 8
          for (int q = 0; q < half; ++q) acc = fmaf(J.ROW[r * half + q], kj[q], acc);
          acc += kj[p];
        } else {
#pragma unroll 8
          for (int q = 0; q < half; ++q) acc = fmaf(J.COL[(r - H) * half + q], kj[half + q], acc);
        }
        val = J.tf32_k ? acc * GF_LOG2E : acc;
      }
      if (is_row) J.Rt[((size_t)b * H + r) * KP + j] = val;
      else J.Ct[((size_t)b * W + (r - H)) * KP + j] = val;
    }
    return;
  }
  // ---- K' role: one thread = 4 channels x 8 latents; the D rows of A are loaded once per thread (4 in flight)
  const int C4 = C >> 2, groups = KP / 8;
  const float4* isc4 = J.in_scale ? reinterpret_cast<const float4*>(J.in_scale + (size_t)b * J.in_ld) : nullptr;
  float4* Kp4 = reinterpret_cast<float4*>(J.Kp + (size_t)b * KP * C);
  for (int item = (blk - J.nvblk - J.npos) * blockDim.x + threadIdx.x; item < C4 * groups; item += J.nkblk * blockDim.x) {
    const int g = item / C4, c4 = item - g * C4;
    const int head = (g * 8) / J.seg, j0 = g * 8 - head * J.seg;      // 8 table columns of one head (seg >= 8): latents j0 .. j0 + 7
    const float* Ah = J.A + (size_t)head * D * LDK;
    float4 acc[8];
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) acc[jj] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (j0 < k) {
      for (int d0 = 0; d0 < D; d0 += 4) {
        float4 a[4];
#pragma unroll
        for (int dd = 0; dd < 4; ++dd) a[dd] = d0 + dd < D ? *reinterpret_cast<const float4*>(Ah + (size_t)(d0 + dd) * LDK + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int dd = 0; dd < 4; ++dd) {
          if (d0 + dd < D) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) {
              if (j0 + jj < k) {
                const float y = ysm[(j0 + jj) * D + d0 + dd];
                acc[jj].x = fmaf(y, a[dd].x, acc[jj].x); acc[jj].y = fmaf(y, a[dd].y, acc[jj].y);
                acc[jj].z = fmaf(y, a[dd].z, acc[jj].z); acc[jj].w = fmaf(y, a[dd].w, acc[jj].w);
              }
            }
          }
        }
      }
    }
    const float4 d = isc4 ? isc4[c4] : make_float4(1.f, 1.f, 1.f, 1.f);
#pragma unroll
    for (int jj = 0; jj < 8; ++jj) {
      float4 r = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j0 + jj < k) {
        const float4 cst = *reinterpret_cast<const float4*>(J.Cst + ((size_t)head * k + j0 + jj) * LDK + c4 * 4);
        r = make_float4((acc[jj].x + cst.x) * d.x, (acc[jj].y + cst.y) * d.y, (acc[jj].z + cst.z) * d.z, (acc[jj].w + cst.w) * d.w);
        if (J.tf32_k) {
          constexpr float kf = GF_TF32_TRUNC_COMP * GF_LOG2E;
          r.x = round_tf32(r.x * kf); r.y = round_tf32(r.y * kf); r.z = round_tf32(r.z * kf); r.w = round_tf32(r.w * kf);
        }
      }
      Kp4[(size_t)(g * 8 + jj) * C4 + c4] = r;
    }
  }
}

static void stage_i_fill(StageIJob& J, const Layout& L, const float* Y, const float* A, const float* Cst, const float* AV, const float* CV,
                         const float* f, float* Kp, float* Vt, float* Rt, float* Ct, const float* in_scale, int in_ld, int tf32_k, int tf32_v) {
  J.Y = Y; J.A = A; J.Cst = Cst; J.AV = AV; J.CV = CV; J.ROW = f + L.f_ROW; J.COL = f + L.f_COL; J.in_scale = in_scale;
  J.Kp = Kp; J.Vt = Vt; J.Rt = Rt; J.Ct = Ct;
  J.CB = f + L.f_CB; J.CBout = nullptr;
  J.H = L.H; J.W = L.W; J.C = L.C; J.k = L.k; J.D = L.D; J.p = L.p; J.KP = L.KP; J.Cout = L.Cout; J.LDK = L.LDK; J.in_ld = in_ld;
  J.tf32_k = tf32_k; J.tf32_v = tf32_v;
  J.heads = L.heads; J.seg = L.heads > 1 ? L.seg : L.KP;       // one head: a single segment of KP columns
  J.nvblk = Vt ? (L.Cout + 255) / 256 : 0;
  J.npos = ((L.H + L.W) * L.KP + 1023) / 1024;
  J.nkblk = ((L.C / 4) * (L.KP / 8) + 255) / 256;
  J.blk_begin = 0;
}

static int stage_i_launch(StageIBatch& batch, int B, cudaStream_t st) {
  int total = 0;
  size_t smem = 0;
  for (int i = 0; i < batch.njobs; ++i) {
    StageIJob& J = batch.job[i];
    J.blk_begin = total;
    total += J.nvblk + J.npos + J.nkblk;
    const size_t need = ((size_t)J.k * J.D + (size_t)J.KP * (J.p + 1)) * sizeof(float);
    if (need > smem) smem = need;
  }
  if (smem > 48 * 1024) { set_error("stage I: k * (D + p + 1) floats exceed 48 KB of shared memory"); return GF_ERR_UNSUPPORTED; }
  stage_i_kernel<<<dim3(B, total), 256, smem, st>>>(batch);
  GF_LAUNCH_OK();
  return GF_OK;
}

int prologue(const Layout& L, const gf_attn_desc* d, const float* Y, const float* key_source, int kdim,
             const float* f, float* ws, cudaStream_t st, const float* in_scale, int in_scale_ld, bool keys_from_xbar, bool with_v) {
  int rc;
  const float* AK = f + (keys_from_xbar ? L.f_AK2 : L.f_AK);
  const float* CK = f + (keys_from_xbar ? L.f_CK2 : L.f_CK);
  // operands of the tcgen05 TF32 contractions are pre-rounded here; the fp32-FMA kernel gets them untouched
  const int tf32 = (!(d->flags & GF_FLAG_FP32_EXACT) && tc_supported(L, d)) ? 1 : 0;
  if (!L.duplex) {
    // simplex: keys from the latents (inner dimension D): the whole of stage I is one launch
    StageIBatch batch;
    batch.njobs = 1;
    stage_i_fill(batch.job[0], L, Y, AK, CK, f + L.f_AV, f + L.f_CV, f, ws + L.w_Kp, ws + L.w_Vt, ws + L.w_Rt, ws + L.w_Ct,
                 in_scale, in_scale_ld, tf32, tf32);
    batch.job[0].CBout = ws + L.w_CB;
    return stage_i_launch(batch, L.B, st);
  }
  // duplex: KPALL [B*k, LDK] = key_source @ AK + CK with key_source = Xbar or the centroids (inner dimension C): tensor cores
  if ((rc = gemm(st, L.B * L.k, L.LDK, kdim, key_source, kdim, false, AK, L.LDK, false, ws + L.w_KPALL, L.LDK, 1.f,
                 CK, L.LDK, L.k, nullptr, tf32 != 0 && kdim >= 64)))
    return rc;
  const int npos = ((L.H + L.W) * L.KP + 1023) / 1024;
  const int nblk = npos + (with_v ? (L.Cout + 255) / 256 : 0) + (L.KP * L.C + 256 * 8 - 1) / (256 * 8);
  finalize_kernel<<<dim3(L.B, nblk), 256, (size_t)L.k * L.D * sizeof(float), st>>>(ws + L.w_KPALL, Y, f + L.f_AV, f + L.f_CV, f + L.f_ROW, f + L.f_COL,
                                                   ws + L.w_Kp, with_v ? ws + L.w_Vt : nullptr, ws + L.w_Rt, ws + L.w_Ct,
                                                   L.H, L.W, L.C, L.k, L.D, L.p, L.KP, L.Cout, L.LDK, tf32, npos, in_scale, in_scale_ld,
                                                   f + L.f_CB, ws + L.w_CB);
  GF_LAUNCH_OK();
  return GF_OK;
}

// duplex pass A tables: M [B,KP,C] and the positional logit tables of the latent queries -- plus V^T of stage T, which
// depends on the latents only (one launch for everything that does not need the centroids)
int duplex_tables(const Layout& L, const gf_attn_desc* d, const float* Y, const float* f, float* ws, cudaStream_t st,
                  const float* in_scale, int in_scale_ld) {
  const int tf32 = tc_centroid_supported(L, d) ? 1 : 0;      // M is an operand of the tcgen05 pass-A kernel: pre-round it
  const int tf32_v = (!(d->flags & GF_FLAG_FP32_EXACT) && tc_supported(L, d)) ? 1 : 0;
  StageIBatch batch;
  batch.njobs = 1;
  stage_i_fill(batch.job[0], L, Y, f + L.f_AM, f + L.f_CM, f + L.f_AV, f + L.f_CV, f, ws + L.w_M, ws + L.w_Vt, ws + L.w_Rt2, ws + L.w_Ct2,
               in_scale, in_scale_ld, tf32, tf32_v);
  return stage_i_launch(batch, L.B, st);
}

// k-means iteration >= 2: pass-A query tables from the previous centroids (inner dimension C: tensor cores)
int duplex_tables_from_centroids(const Layout& L, const gf_attn_desc* d, const float* cen, const float* Y, const float* f, float* ws,
                                 cudaStream_t st, const float* in_scale, int in_scale_ld) {
  int rc;
  const int tf32 = tc_centroid_supported(L, d) ? 1 : 0;
  // fp32 product: the queries feed a softmax over the n grid cells, and the k-means loop feeds its own output back -- a TF32 error
  // here is amplified by every further iteration (measured: image rel-RMS 3.2e-3 with TF32 against 4.7e-4 for a plain duplex layer)
  if ((rc = gemm(st, L.B * L.k, L.LDK, L.C, cen, L.C, false, f + L.f_ACQ, L.LDK, false, ws + L.w_MALL, L.LDK, 1.f,
                 f + L.f_CM, L.LDK, L.k, nullptr, false)))
    return rc;
  const int npos = ((L.H + L.W) * L.KP + 1023) / 1024;
  const int nblk = npos + (L.KP * L.C + 256 * 8 - 1) / (256 * 8);
  finalize_kernel<<<dim3(L.B, nblk), 256, 0, st>>>(ws + L.w_MALL, Y, nullptr, nullptr, f + L.f_ROW, f + L.f_COL,
                                                   ws + L.w_M, nullptr, ws + L.w_Rt2, ws + L.w_Ct2,
                                                   L.H, L.W, L.C, L.k, L.D, L.p, L.KP, L.Cout, L.LDK, tf32, npos, in_scale, in_scale_ld,
                                                   nullptr, nullptr);
  GF_LAUNCH_OK();
  return GF_OK;
}

// g_img2ltnt: Y2[r, :] = LN(Y[r, :]) * (1 + Cen[r, :] . WI2L + BI2L), one warp per latent row r = b * k + j
__global__ void __launch_bounds__(128) img2ltnt_kernel(const float* __restrict__ Y, const float* __restrict__ cen, const float* __restrict__ Wi,
                                                       const float* __restrict__ bi, float* __restrict__ Y2, int rows, int C, int D) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.x * 4 + warp;
  if (r >= rows) return;
  const float* y = Y + (size_t)r * D;
  float s = 0.f, ss = 0.f;
  for (int d0 = lane; d0 < D; d0 += 32) s += y[d0];
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mu = s / (float)D;
  for (int d0 = lane; d0 < D; d0 += 32) { const float t = y[d0] - mu; ss = fmaf(t, t, ss); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float rstd = rsqrtf(ss / (float)D + 1e-8f);
  const float* c = cen + (size_t)r * C;
  for (int d0 = lane; d0 < D; d0 += 32) {
    float acc = bi[d0];
    for (int cc = 0; cc < C; ++cc) acc = fmaf(c[cc], Wi[(size_t)cc * D + d0], acc);      // c[cc]: warp-uniform (one transaction)
    Y2[(size_t)r * D + d0] = (y[d0] - mu) * rstd * (1.f + acc);
  }
}

int img2ltnt(const Layout& L, const float* Y, const float* cen, const float* f, float* ws, cudaStream_t st) {
  const int rows = L.B * L.k;
  img2ltnt_kernel<<<(rows + 3) / 4, 128, 0, st>>>(Y, cen, f + L.f_WI2L, f + L.f_BI2L, ws + L.w_Y2, rows, L.C, L.D);
  GF_LAUNCH_OK();
  return GF_OK;
}

// Stage I of several layers (same batch size, same latents or not) in ONE launch: simplex layers get their keys, V^T and
// positional tables; duplex layers their pass-A query tables and V^T (everything that does not depend on the activations).
int prologue_batch(int n, const Layout* Ls, const gf_attn_desc* const* ds, const float* const* Ys, const float* const* fs, float* const* wss,
                   const gf_attn_postop* const* posts, cudaStream_t st) {
  int done = 0;
  while (done < n) {
    StageIBatch batch;
    batch.njobs = 0;
    const int B = Ls[done].B;
    while (done < n && batch.njobs < STAGE_I_MAX_JOBS && Ls[done].B == B) {
      const Layout& L = Ls[done];
      const gf_attn_desc* d = ds[done];
      const float* f = fs[done];
      float* ws = wss[done];
      const gf_attn_postop* post = posts ? posts[done] : nullptr;
      const float* isc = post ? post->in_scale : nullptr;
      const int isc_ld = post ? post->in_scale_ld : 0;
      const int tf32_t = (!(d->flags & GF_FLAG_FP32_EXACT) && tc_supported(L, d)) ? 1 : 0;
      StageIJob& J = batch.job[batch.njobs++];
      if (L.duplex)
        stage_i_fill(J, L, Ys[done], f + L.f_AM, f + L.f_CM, f + L.f_AV, f + L.f_CV, f, ws + L.w_M, ws + L.w_Vt, ws + L.w_Rt2, ws + L.w_Ct2,
                     isc, isc_ld, tc_centroid_supported(L, d) ? 1 : 0, tf32_t);
      else {
        stage_i_fill(J, L, Ys[done], f + L.f_AK, f + L.f_CK, f + L.f_AV, f + L.f_CV, f, ws + L.w_Kp, ws + L.w_Vt, ws + L.w_Rt, ws + L.w_Ct,
                     isc, isc_ld, tf32_t, tf32_t);
        J.CBout = ws + L.w_CB;
      }
      ++done;
    }
    int rc = stage_i_launch(batch, B, st);
    if (rc) return rc;
  }
  return GF_OK;
}

}  // namespace gf
