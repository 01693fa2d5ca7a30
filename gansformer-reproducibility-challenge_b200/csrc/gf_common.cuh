// gf_common.cuh -- shared host/device definitions for libgf_attn (sm_100a only).
//
// Buffer layouts are the ones restated in oracle/folded.py (stage W / I / T); keep the two in sync.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <math.h>
#include "../../include/gf_attn.h"

namespace gf {

// ---- thread-local error reporting -----------------------------------------------------------------
void set_error(const char* fmt, ...);
void set_path(int path);
void set_centroid_path(int path);
void note_launch();

#define GF_CUDA_OK(expr)                                                                         \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      gf::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));       \
      return GF_ERR_CUDA;                                                                        \
    }                                                                                            \
  } while (0)

#define GF_LAUNCH_OK()                                                                           \
  do {                                                                                           \
    cudaError_t _e = cudaGetLastError();                                                         \
    if (_e != cudaSuccess) {                                                                     \
      gf::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e));   \
      return GF_ERR_CUDA;                                                                        \
    }                                                                                            \
    gf::note_launch();                                                                           \
  } while (0)

// ---- layout of the folded-weight buffer and of the per-call workspace -----------------------------
// All offsets in floats, each region 64-float (256 B) aligned.
struct Layout {
  int B, H, W, C, k, D, p, KP, Cout, LDK, n, duplex;
  // folded buffer (stage W)
  size_t f_AK, f_CK, f_AV, f_CV, f_ROW, f_COL;        // simplex + duplex
  size_t f_WV2, f_BV2, f_AM, f_CM;                    // duplex only
  size_t f_QFOLD, f_KCONST, f_MFOLD, f_QCONST;        // scratch of stage W
  size_t f_total;
  // workspace (stage I/T)
  size_t w_KPALL, w_Kp, w_Vt, w_Rt, w_Ct;             // keys / values / positional logit tables
  size_t w_NSCALE, w_NSHIFT, w_NPART;                 // instance/batch norm statistics
  size_t w_MALL, w_M, w_Rt2, w_Ct2, w_PART, w_XBAR;   // duplex pass A
  size_t f_AK2, f_CK2;                                // duplex: keys straight from Xbar (Wv2 and bv2 folded into AK / CK)
  size_t f_CB, w_CB;                                  // bo (+1 on the gain half): the part of the control signal attention dropout must NOT scale
  size_t f_ACQ, f_WI2L, f_BI2L;                       // kmeans_iters > 1: centroid -> pass-A query table; g_img2ltnt: centroid -> latent gain
  size_t w_CEN, w_Y2;                                 // scratch centroids [B,k,C] (caller passed none), modulated latents [B,k,D]
  int iters, img2ltnt;
  int heads, seg;                                     // num_heads; per-head segment of the KP "latent" columns (KP = heads * seg, seg >= k)
  size_t w_total;
  int nsplit_norm, nsplit_cen;
};

// SM count of the current device (B200: 148), queried once per process; grids and split models are sized from it.
inline int num_sms() {
  static int v = -1;
  if (v < 0) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) v = n;
    else return 148;          // no device visible (host-only layout queries): the B200 figure, not cached
  }
  return v;
}

// ---- attention dropout (att_dp, training): counter-based Philox4x32-10, reproducible on the CPU (oracle/philox.py) ----------
// One call yields the keep decisions of 4 consecutive table columns of one token:
//   counter = (global token index b * n + t, column block j / 4, salt (per layer), 0x5eed),  key = seed (lo, hi)
//   keep_j  = word_j >= thr,  thr = round(p * 2^32);  kept probabilities are scaled by 1 / (1 - p).
struct DropoutArgs {
  const unsigned long long* state;   // device: {seed, step counter} -- read at run time, so a replayed CUDA graph draws fresh masks
  uint32_t thr;                      // 0 = dropout off
  uint32_t salt;                     // distinguishes the layers of a network
  float scale;                       // 1 / (1 - p)
};
#ifdef __CUDACC__
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// multipliers (0 or 1/(1-p)) of columns 4q .. 4q+3 of global token `tok`
__device__ __forceinline__ void dropout_mult4(const DropoutArgs& D, unsigned long long seed, unsigned long long step, uint32_t tok, int q, float mk[4]) {
  uint32_t w[4];
  philox4x32_10(tok, (uint32_t)q | ((uint32_t)step << 8), D.salt ^ (uint32_t)(step >> 24), 0x5eedu, (uint32_t)seed, (uint32_t)(seed >> 32), w);
#pragma unroll
  for (int i = 0; i < 4; ++i) mk[i] = w[i] >= D.thr ? D.scale : 0.f;
}
#endif

inline size_t align64(size_t x) { return (x + 63) & ~size_t(63); }
inline int pad_k(int k) { return k <= 16 ? 16 : 32; }

// Fills L; returns GF_OK or an error (message set).
int make_layout(const gf_attn_desc* d, Layout* L);
int check_device();          // GF_OK on a compute-capability-10.x device, an error otherwise (gf_api.cu)

// ---- stage W / I kernels (gf_fold.cu) ---------------------------------------------------------------
int fold_weights(const Layout& L, const gf_attn_desc* d, const gf_attn_weights* w, float* folded, cudaStream_t st);
// key_source: Y [B*k, D] (simplex) or centroids [B*k, C] (duplex); kdim = D or C.
int prologue(const Layout& L, const gf_attn_desc* d, const float* Y, const float* key_source, int kdim,
             const float* folded, float* ws, cudaStream_t st, const float* in_scale = nullptr, int in_scale_ld = 0,
             bool keys_from_xbar = false, bool with_v = true);
int prologue_batch(int n, const Layout* Ls, const gf_attn_desc* const* ds, const float* const* Ys, const float* const* fs, float* const* wss,
                   const gf_attn_postop* const* posts, cudaStream_t st);
int duplex_tables_from_centroids(const Layout& L, const gf_attn_desc* d, const float* cen, const float* Y, const float* f, float* ws,
                                 cudaStream_t st, const float* in_scale, int in_scale_ld);
int img2ltnt(const Layout& L, const float* Y, const float* cen, const float* f, float* ws, cudaStream_t st);
int duplex_tables(const Layout& L, const gf_attn_desc* d, const float* Y, const float* folded, float* ws, cudaStream_t st,
                  const float* in_scale = nullptr, int in_scale_ld = 0);
// C[M,N] = alpha * opA(A) opB(B) + E[(m % emod), n] + v[n]
int gemm(cudaStream_t st, int M, int N, int K, const float* A, int lda, bool ta, const float* B, int ldb, bool tb,
         float* Cm, int ldc, float alpha, const float* E = nullptr, int lde = 0, int emod = 1, const float* v = nullptr,
         bool allow_tf32 = false);
// tcgen05 TF32 version for dense row-major operands (gf_tc_gemm.cu); gemm() routes to it when allow_tf32 and the shape fits
bool gemm_tc_ok(int M, int N, int K, const float* A, const float* B, const float* Cm, int ldc);
int gemm_tc(cudaStream_t st, int M, int N, int K, const float* A, const float* B, float* Cm, int ldc, float alpha,
            const float* E, int lde, int emod, const float* v);

// ---- stage T kernels ----------------------------------------------------------------------------------
int token_pass_simt(const Layout& L, const gf_attn_desc* d, const float* X, float* Xout, float* att, float* ws, const gf_attn_postop* post, cudaStream_t st);
// postop -> DropoutArgs (thr = 0 when off); GF_ERR_INVALID on a bad probability / missing state
int dropout_args(const gf_attn_postop* post, DropoutArgs* out);
int norm_stats(const Layout& L, const gf_attn_desc* d, const float* X, float* ws, cudaStream_t st);
int centroid_pass_simt(const Layout& L, const gf_attn_desc* d, const float* X, float* ws, cudaStream_t st,
                       const float* in_scale = nullptr, int in_scale_ld = 0);
// pass-A partials (per split: acc [KP][C], running max and denominator) of the CUDA-core kernel on the given tables, into `part`
int centroid_partials_simt(const Layout& L, const float* X, const float* M, const float* Rt, const float* Ct, float* part, cudaStream_t st);
// Xbar = merge of the split partials in ws (times the load-side scale, when given); into ws + w_XBAR unless `xbar` is given;
// lse [B,k] (nullable) = log of each latent's softmax denominator
int centroid_merge(const Layout& L, float* ws, cudaStream_t st, const float* in_scale = nullptr, int in_scale_ld = 0,
                   float* xbar = nullptr, float* lse = nullptr);
// tcgen05 duplex pass A (gf_tc_cen.cu): partials into ws (same format as the CUDA-core kernel), then centroid_merge
bool tc_centroid_supported(const Layout& L, const gf_attn_desc* d);
// in_scale: only used when the split count is 1 and the kernel writes the normalised Xbar itself (no merge kernel)
int centroid_pass_tc(const Layout& L, const gf_attn_desc* d, const float* X, float* ws, cudaStream_t st,
                     const float* in_scale = nullptr, int in_scale_ld = 0);
// tcgen05 / TMA path (gf_tc.cu).  tc_supported() says whether the shape is served by it.
bool tc_supported(const Layout& L, const gf_attn_desc* d);
int token_pass_tc(const Layout& L, const gf_attn_desc* d, const float* X, float* Xout, float* att, float* ws, const gf_attn_postop* post, cudaStream_t st);

}  // namespace gf
