/*
 * gf_attn.h -- C ABI of the B200-native GANsformer bipartite-attention hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  The reference has no FFI for this path: its attention block
 * is Python/TensorFlow graph code, expected at src/training/network.py (transformer_layer, integrate,
 * att_norm, dense_layer, get_positional_embeddings) -- NOT present in the reference checkout
 * (/root/reference/.SUBMODULES.json:2 reports "bytes": 0), so no file:line can be cited; the only
 * reference files on disk are LICENSE and src/Dockerfile (:7 pins tensorflow 1.14).  Each entry point
 * below names the reference function it replaces.  INTEGRATION.md shows the ctypes stub a maintainer of
 * the reference would add inside transformer_layer().
 *
 * Conventions
 *   - plain C, no torch / CUDA-runtime types in signatures; `stream` is a cudaStream_t passed as void*.
 *   - every pointer is a DEVICE pointer unless named host_*; the library never allocates or frees
 *     device memory and never synchronises; all work is enqueued on `stream`.
 *   - activations are channels-last fp32: X[B][H][W][C]  (== [B*n][C] row-major, n = H*W).
 *   - return value: GF_OK (0) or a negative gf_status; gf_last_error() gives a thread-local message.
 *   - unsupported shape / device => error.  There is no CPU path and no fallback of any kind.
 */
#ifndef GF_ATTN_H_
#define GF_ATTN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_ATTN_ABI_VERSION 2

typedef enum gf_status {
  GF_OK = 0,
  GF_ERR_INVALID = -1,      /* bad descriptor / null pointer */
  GF_ERR_UNSUPPORTED = -2,  /* valid request this build has no kernel for */
  GF_ERR_CUDA = -3,         /* CUDA runtime / driver error (message has the string) */
  GF_ERR_WORKSPACE = -4     /* workspace or folded buffer too small */
} gf_status;

/* att_norm(): which statistics normalise X before modulation */
enum { GF_NORM_NONE = 0, GF_NORM_LAYER = 1, GF_NORM_INSTANCE = 2, GF_NORM_BATCH = 3 };
/* integrate(): how the control signal modulates X */
enum { GF_INT_MUL = 0, GF_INT_ADD = 1, GF_INT_BOTH = 2 };
/* desc.flags */
enum {
  GF_FLAG_FP32_EXACT = 1,   /* force the CUDA-core fp32-FMA kernel (tight-tolerance mode); default = tcgen05 TF32 */
  GF_FLAG_CENTROIDS_IN = 2, /* duplex: skip pass A, take centroids_inout as input (iterative=True upstream) */
  GF_FLAG_TABLES_READY = 4, /* duplex: the pass-A query tables and V^T are already in ws (gf_attn_prologue_batch ran for this layer) */
  GF_FLAG_CENTROIDS_INIT = 16, /* duplex: `iterative` -- centroids_inout holds the previous attention layer's centroids on entry; the
                               first k-means iteration takes its queries from them (through wcq) instead of from the latents; on
                               return it holds this layer's centroids */
  GF_FLAG_IMG2LTNT = 8      /* duplex: g_img2ltnt -- before pass B the latents are modulated by the centroids,
                               Y <- LN(Y) (1 + dense(Cen, wi2l) + bi2l); values of pass B from the modulated latents */
};
/* which kernel family served the last forward on this thread (gf_attn_last_path) */
enum { GF_PATH_NONE = 0, GF_PATH_SIMT_FP32 = 1, GF_PATH_TCGEN05_TF32 = 2 };

/* Shape/config of one attention layer call.  Mirrors the kwargs of the reference's
 * transformer_layer(dim, pos_dim, from_tensor, to_tensor, from_len, to_len, num_heads, integration, norm, kmeans...) */
typedef struct gf_attn_desc {
  int32_t B, H, W, C;   /* X[B,H,W,C]; from_len = H*W, dim = C */
  int32_t k, D;         /* Y[B,k,D]; to_len = k latents of size D */
  int32_t heads;        /* num_heads; this build: 1 */
  int32_t norm;         /* GF_NORM_* */
  int32_t integration;  /* GF_INT_* */
  int32_t pos_dim;      /* width of the positional embeddings; 0 = use_pos False */
  int32_t duplex;       /* 0 = simplex (latents -> image); n >= 1 = duplex (kmeans) with n k-means iterations (kmeans_iters):
                           iteration i >= 2 takes its queries from the previous centroids through wcq */
  int32_t flags;        /* GF_FLAG_* */
} gf_attn_desc;

/* Optional fusion of what surrounds the attention block inside the reference's synthesis layer:
 *   load side :  x_in = X * in_scale[b,c]            (StyleGAN2 demodulation of the preceding convolution's output)
 *   store side:  x'' = act(x' + noise[b*noise_bstride + t] * (*strength) + bias[c]) * gain * post_scale[b,c]
 *                (noise input + fused_bias_act, then the style modulation of the NEXT convolution's input)
 * in_scale must be given to BOTH gf_attn_prologue_ex (it is folded into K') and gf_attn_simplex_fwd_ex; gf_attn_duplex_fwd_ex
 * additionally folds it into the pass-A query matrix and the centroid means (the latents see x_in too).
 * The scales need norm layer/none; every member may be NULL. */
typedef struct gf_attn_postop {
  const float* bias;         /* [C] or NULL */
  const float* noise;        /* [H*W] (noise_bstride = 0: shared by the batch) or [B][H*W]; NULL = no noise */
  const float* strength;     /* device scalar; NULL = 1 */
  long long noise_bstride;
  int32_t act;               /* 0 linear, 1 leaky-ReLU(0.2) */
  float gain;
  const float* in_scale;     /* [B][in_scale_ld] rows of C floats, 16-byte aligned rows; NULL = 1 */
  const float* post_scale;   /* [B][post_scale_ld]; NULL = 1 */
  int32_t in_scale_ld, post_scale_ld;
  /* fused tRGB (the 1x1 modulated convolution, no demodulation, that follows the last layer of a resolution block):
   *   rgb_out[b][o][t] = sum_c x''[b,t,c] * rgb_w[b][o][c] + rgb_bias[o],  o < 3,  x'' = the layer output BEFORE post_scale.
   * rgb_w [B][3][C] contiguous (weight * style * 1/sqrt(C) per sample), 16-byte aligned; rgb_bias [3] or NULL; rgb_out [B][3][H*W]
   * planar.  All NULL = off.  Served by the tcgen05 path only (gf_attn_tc_eligible) for C <= 256, or C = 512 with k <= 16; other
   * shapes and the CUDA-core path return UNSUPPORTED. */
  const float* rgb_w;
  const float* rgb_bias;
  float* rgb_out;
  /* attention dropout (att_dp of transformer_layer; training only): every probability of the k-softmax is dropped with probability
   * att_dp and the survivors are scaled by 1 / (1 - att_dp).  The mask is Philox4x32-10 of (token, column block, dp_salt, step) keyed
   * by the seed; dp_state points to DEVICE memory {uint64 seed, uint64 step} read when the kernel runs (bump `step` on the device
   * between training steps: a replayed CUDA graph then draws fresh masks).  Both kernel families serve it with the same mask (the
   * tcgen05 kernel drops the probabilities before they become GEMM2's operand); the attention map output is the probabilities
   * BEFORE dropout.  att_dp = 0 or dp_state = NULL: off.
   * Duplex layers: only pass B's softmax over the k latents is dropped (same Philox stream, token = b * n + t); pass A's softmax over
   * the n grid cells, which builds the centroids, never is. */
  float att_dp;
  uint32_t dp_salt;
  const unsigned long long* dp_state;
} gf_attn_postop;

/* Raw (un-scaled) parameters of one layer, each [fan_in, fan_out] row-major; equalised-LR scaling
 * (1/sqrt(fan_in), reference: get_weight/dense_layer) is applied by the library.  The *2 / wkc
 * members are only read when desc.duplex; wpq/wpk/pos_latent (and wpq2/wpk2) only when pos_dim>0. */
typedef struct gf_attn_weights {
  const float *wq, *bq, *wpq;      /* [C,C] [C] [p,C]   query side (grid)            */
  const float *wk, *bk, *wpk;      /* [D,C] [C] [p,C]   key side (latents; wk unused in duplex) */
  const float *wv, *bv;            /* [D,C] [C]         values (latents)             */
  const float *wo, *bo;            /* [C,Cout] [Cout]   integrate()'s dense, Cout = C or 2C ("both") */
  const float *pos_latent;         /* [k,p]             learned latent positional embedding */
  const float *wq2, *bq2, *wpq2;   /* [D,C] [C] [p,C]   duplex pass A: latent queries */
  const float *wk2, *bk2, *wpk2;   /* [C,C] [C] [p,C]   duplex pass A: grid keys      */
  const float *wv2, *bv2;          /* [C,C] [C]         duplex pass A: grid values    */
  const float *wkc;                /* [C,C]             centroid -> key               */
  const float *wcq;                /* [C,C]             centroid -> query of k-means iterations >= 2 (read when desc.duplex > 1) */
  const float *wi2l, *bi2l;        /* [C,D] [D]         centroid -> latent gain (read with GF_FLAG_IMG2LTNT) */
} gf_attn_weights;

/* Library / device introspection. */
int gf_attn_abi_version(void);
const char* gf_last_error(void);
int gf_attn_last_path(void);
/* same for the duplex pass-A (centroid) kernel of the last gf_attn_duplex_fwd on this thread */
int gf_attn_last_centroid_path(void);
/* Number of kernels this library has launched in this process (all threads); bench.py reports the delta. */
long long gf_attn_launch_count(void);

/* 1 when gf_attn_simplex_fwd / stage T of this layer runs on the tcgen05 (TF32) kernel, 0 when the CUDA-core kernel serves it
 * (GF_FLAG_FP32_EXACT, instance / batch norm, C not in {64,128,256,512}, ragged n); negative gf_status on a bad descriptor. */
int gf_attn_tc_eligible(const gf_attn_desc* desc);

/* Debug aid for the bring-up probes (tools/): float offsets {w_PART, w_XBAR, nsplit_cen, KP, w_M, w_Rt2, w_Ct2, w_total} of the workspace. */
int gf_attn_debug_layout(const gf_attn_desc* desc, long long* out, int n);

/* Size in floats of the folded-weight buffer (stage W output + its scratch). */
int gf_attn_folded_floats(const gf_attn_desc* desc, size_t* out_floats);

/* Stage W -- replaces the weight-only part of dense_layer()/get_weight(): folds Wq,Wk,Wpq,Wpk,Wo,...
 * into the small matrices the per-image prologue consumes.  Run once per weight update. */
int gf_attn_fold_weights(const gf_attn_desc* desc, const gf_attn_weights* weights, float* folded, void* stream);

/* Size in bytes of the per-call workspace for batch desc->B. */
int gf_attn_workspace_bytes(const gf_attn_desc* desc, size_t* out_bytes);

/* Stage I -- replaces the K/V dense layers + get_positional_embeddings() of transformer_layer():
 * per image builds K' [B,KP,C], V^T [B,Cout,KP] and the separable positional-logit tables in `ws`.
 * Simplex: keys from Y.  Duplex: called internally by gf_attn_duplex_fwd after pass A. */
int gf_attn_prologue(const gf_attn_desc* desc, const float* Y, const float* folded, void* ws, void* stream);

/* gf_attn_prologue with the load-side fusion: K' is additionally scaled by post->in_scale (post may be NULL). */
int gf_attn_prologue_ex(const gf_attn_desc* desc, const float* Y, const float* folded, void* ws, const gf_attn_postop* post, void* stream);

/* Stage I of n layers in ONE launch (same batch size): everything that depends on the latents only -- for a simplex layer
 * what gf_attn_prologue_ex builds, for a duplex layer the pass-A query tables and V^T (then call gf_attn_duplex_fwd_ex with
 * GF_FLAG_TABLES_READY).  The reference's G_synthesis calls transformer_layer once per layer with the same latents; the
 * per-layer K/V dense layers it runs each time are batched here.  posts may be NULL, and so may any posts[i]. */
int gf_attn_prologue_batch(int n, const gf_attn_desc* const* descs, const float* const* Y, const float* const* folded, void* const* ws,
                           const gf_attn_postop* const* posts, void* stream);

/* Stage T -- replaces the body of transformer_layer() + integrate() + att_norm() for simplex attention:
 * one read of X, one write of Xout (may alias X).  att (nullable) receives softmax probabilities [B,n,k].
 * Requires gf_attn_prologue() on the same ws/stream first. */
int gf_attn_simplex_fwd(const gf_attn_desc* desc, const float* X, float* Xout, float* att, void* ws, void* stream);

/* Same as gf_attn_simplex_fwd with the fused noise + bias + activation epilogue (post may be NULL). */
int gf_attn_simplex_fwd_ex(const gf_attn_desc* desc, const float* X, float* Xout, float* att, void* ws,
                           const gf_attn_postop* post, void* stream);

/* Duplex (kmeans) layer: pass A (latents attend to the grid, softmax over n, centroids [B,k,C]) then
 * prologue with keys from the centroids, then stage T.  centroids_inout: output (and input when
 * GF_FLAG_CENTROIDS_IN); may be NULL when the caller does not need the centroids -- the keys are then built straight from
 * the attention-weighted means (the centroid projection is folded into the key projection at stage W). */
int gf_attn_duplex_fwd(const gf_attn_desc* desc, const float* X, const float* Y, const float* folded,
                       float* Xout, float* att, float* centroids_inout, void* ws, void* stream);

int gf_attn_duplex_fwd_ex(const gf_attn_desc* desc, const float* X, const float* Y, const float* folded,
                          float* Xout, float* att, float* centroids_inout, void* ws, const gf_attn_postop* post, void* stream);

/* Per-(b,c) statistics for GF_NORM_INSTANCE / GF_NORM_BATCH, written into ws by a reduction pass over X
 * (called internally by the forward entry points; exported for tests). */
int gf_attn_norm_stats(const gf_attn_desc* desc, const float* X, void* ws, void* stream);

/* Backward of stage T for simplex layers with norm layer/none (SURVEY row f2) -- replaces what TensorFlow's autodiff derives
 * for transformer_layer()/integrate().  Inputs: X and the incoming gradient dOut [B,n,C]; the per-image tables of stage I in
 * the workspace layout (Kp [B,KP,C], Vt [B,Cout,KP], Rt [B,H,KP] with -inf in the padded latents, Ct [B,W,KP]; KP = 16 for
 * k <= 16, else 32), fp32, un-rounded.  Outputs: dX [B,n,C]; dS [B,n,KP] = gradient w.r.t. the logits; P [B,n,KP] = the
 * probabilities; dCtl [B,n,Cout] = gradient w.r.t. the control signal (gain half | bias half).  The reductions over the
 * tokens that remain are plain batched products the caller runs with its GEMM library:
 *   dKp[b] = dS[b]^T X[b],  dVt[b] = dCtl[b]^T P[b],  dRt[b,h,:] = sum_w dS[b,h,w,:],  dCt[b,w,:] = sum_h dS[b,h,w,:]. */
int gf_attn_simplex_bwd(const gf_attn_desc* desc, const float* X, const float* dOut, const float* Kp, const float* Vt,
                        const float* Rt, const float* Ct, float* dX, float* dS, float* P, float* dCtl, void* stream);

/* gf_attn_simplex_bwd with attention dropout: the same (att_dp, dp_salt, dp_state) as the forward call regenerate the mask;
 * Stage T of a duplex layer is differentiated here too: the kernel consumes the tables only, so the caller passes a descriptor with
 * duplex = 0 and tables whose keys come from the centroids (and values from the modulated latents with g_img2ltnt);
 * P then receives the probabilities AFTER dropout q (what dVt = dCtl^T P needs), dS the gradient w.r.t. the logits.
 * cb [Cout] = bo (+1 on the gain half): the constants dropout does not scale -- ctl = sum_j q_j (Vt_j - cb) + cb; the caller adds
 * dcb = sum_tokens dCtl * (1 - sum_j q_j) to the gradient of bo.  cb may be NULL when att_dp == 0. */
int gf_attn_simplex_bwd_ex(const gf_attn_desc* desc, const float* X, const float* dOut, const float* Kp, const float* Vt,
                           const float* Rt, const float* Ct, float* dX, float* dS, float* P, float* dCtl,
                           float att_dp, uint32_t dp_salt, const unsigned long long* dp_state, const float* cb, void* stream);

/* Backward of duplex pass A, part 1 -- recomputes, in fp32 on the CUDA cores, what the forward's pass A computed from the caller's
 * differentiable tables: per image, latent j < k, token t,
 *   Sa[j,t] = x_t.M[j] + Rt2[h(t),j] + Ct2[w(t),j],   A = softmax over the n tokens of Sa,   Xbar = A X,
 * with M [B,KP,C], Rt2 [B,H,KP] (-inf in the padded latents), Ct2 [B,W,KP] in the workspace layout (1/sqrt(C) folded in, KP = 16 for
 * k <= 16, else 32).  Outputs: Xbar [B,k,C] and lse [B,k] = log sum_t exp Sa[j,t].  desc.duplex >= 1; ws = a workspace of
 * gf_attn_workspace_bytes(desc) (its pass-A partials are the scratch).  Split partials are merged in a fixed order: deterministic. */
int gf_attn_centroid_recompute(const gf_attn_desc* desc, const float* X, const float* M, const float* Rt2, const float* Ct2,
                               float* Xbar, float* lse, void* ws, void* stream);

/* Backward of duplex pass A, part 2 -- given dXbar [B,k,C] and what gf_attn_centroid_recompute returned for the same tables:
 *   A = exp(Sa - lse),  dA[j,t] = x_t.dXbar[j],  r_j = Xbar[j].dXbar[j],  dSa = A (dA - r),
 *   dX [B,n,C] += dSa.M + A.dXbar   (accumulated in place: pass the stage-T activation gradient),
 *   dSa [B,n,KP] written (0 in the padded latents).
 * The reductions over the tokens that remain are the caller's: dM[b] = dSa[b]^T X[b], dRt2[b,h,:] = sum_w dSa[b,h,w,:],
 * dCt2[b,w,:] = sum_h dSa[b,h,w,:].  No host synchronisation (capturable in a CUDA graph). */
int gf_attn_centroid_bwd(const gf_attn_desc* desc, const float* X, const float* M, const float* Rt2, const float* Ct2,
                         const float* lse, const float* Xbar, const float* dXbar, float* dX, float* dSa, void* stream);

/* The dropout multipliers themselves, mask [B, H*W, KP] (0 or 1 / (1 - att_dp); KP = 16 for k <= 16, else 32; columns of a
 * multi-head layer: head * seg + j): what the fused kernels apply.  For the composite training path and for tests. */
int gf_attn_dropout_mask(const gf_attn_desc* desc, float att_dp, uint32_t dp_salt, const unsigned long long* dp_state, float* mask, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GF_ATTN_H_ */
