/*
 * gecco_b200 — C ABI of the B200 (sm_100a) implementation of gecco-torch's
 * reverse-diffusion sampling path.
 *
 * The reference (cvlab-epfl/gecco, gecco-torch) has no FFI of its own: the path
 * sits behind plain Python nn.Module calls (SURVEY.md §8b).  This header is the
 * boundary a maintainer binds instead of the ATen call sites listed in
 * SURVEY.md §2.2; each entry point cites the reference code it replaces
 * (paths relative to gecco-torch/src/gecco_torch/).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless named host_*; the caller (torch)
 *     owns all memory, the library never allocates or frees user-visible buffers;
 *   - every launch function takes the CUDA stream as a void* (cudaStream_t), is
 *     asynchronous, does no host synchronisation and is CUDA-graph capturable;
 *   - every export returns 0 on success or a negative GECCO_ERR_* code;
 *     gecco_last_error() returns the text of the last failure on this thread;
 *   - there is no CPU fallback: a device that is not sm_100 is an error.
 */
#ifndef GECCO_B200_H
#define GECCO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GECCO_OK 0
#define GECCO_ERR_INVALID (-1) /* bad argument / unsupported shape */
#define GECCO_ERR_CUDA (-2)    /* CUDA runtime or driver error      */
#define GECCO_ERR_DEVICE (-3)  /* not an sm_100 device              */

#define GECCO_ABI_VERSION 1

int gecco_abi_version(void);
const char* gecco_last_error(void);
/* Checks that `device` is sm_100 and resolves the driver entry points. */
int gecco_init(int device);

/* Tuning switches.  "gemm_pairs" (default 1): use the CTA-pair (cta_group::2) GEMM where it applies;
 * "graphs" (default 1, or GECCO_GRAPHS=0 in the environment): gecco_sample captures its launch sequence into a
 * CUDA graph on the first call with a given argument set and replays it afterwards;
 * "anorm" (default 1, or GECCO_ANORM=0): the engine normalises (AdaGN) inside the consuming projection where the shape
 * allows (gecco_anorm) instead of folding the normalisation into per-cloud weights. */
int gecco_set_option(const char* name, int value);

/* ------------------------------------------------------------------------
 * Dense projection on the tcgen05 tensor cores.
 *   out[m, n] = epilogue( sum_k a[m, k] * w[wrow(m) + n, k] )
 * a: bf16 [M, K] row-major (lda elements), w: bf16 [*, K] row-major (ldw).
 * Replaces every nn.Linear / F.linear on the path: kv_proj
 * (models/set_transformer.py:49), the in/out projections of nn.MultiheadAttention
 * (:90,112), MLP (models/mlp.py:5-39) and img_feature_proj (models/ray.py:52-55).
 * Epilogue, applied in this order on the fp32 accumulator:
 *   + bias[cloud*bias_stride + n]                     (bias may be NULL)
 *   + xyz embed: sum_j c_in(sigma)*geom[point,j]*wx[n,j]  (geom may be NULL; models/ray.py:99,113)
 *   Gaussian activation (exp(-z^2/(2 alpha^2)) - 0.7)/0.28 when act != 0 (models/activation.py:17-24)
 *   + res[m, n]                                       (res may be NULL; residual adds set_transformer.py:164,166)
 *   per (cloud, 12-channel group) sum / sum of squares of the result added into
 *   stats (double [clouds][n_out/12][2]) for the next AdaGN (models/normalization.py:36-44)
 * and written as fp32 (out_f32) and/or bf16 (out_bf16).
 * Rows are grouped in clouds of rows_per_cloud rows of which the first valid_rows
 * are real points (the rest is padding, excluded from stats).
 * ------------------------------------------------------------------------ */
/* AdaGN applied to the A operand inside the projection (models/normalization.py:36-44 in front of an nn.Linear,
 * set_transformer.py:49,112,162,165): when stats != NULL, `a` is the UN-normalised bf16 tensor x [M, K] and the kernel
 * multiplies by
 *     bf16( scale_b(t)[k] * (x[m,k] - mean[b,g]) * rstd[b,g] + bias_b(t)[k] )
 * (fp32 arithmetic, one rounding), rewriting each operand tile in shared memory before the tensor core reads it.
 * mean / rstd come from stats (double [clouds][K/stat_gs][2] sums over the valid rows, as written by a producing
 * epilogue), groups = number of normalisation groups, t[cloud*t_stride] the noise embedding, scale/bias the two
 * nn.Linear(1, K) of AdaGN.  Supported where gecco_gemm_anorm_supported() says so (CTA-pair kernel shapes). */
typedef struct gecco_anorm {
  const double* stats; int32_t stat_gs; int32_t groups; float eps;
  const float* t; int32_t t_stride;
  const float* scale_w; const float* scale_b; const float* bias_w; const float* bias_b;
} gecco_anorm;

typedef struct gecco_gemm_args {
  const void* a;   int64_t lda;
  const void* w;   int64_t ldw;
  int32_t m, n_out, k;
  int32_t rows_per_cloud;   /* > 0, multiple of 32 */
  int32_t valid_rows;       /* <= rows_per_cloud */
  int32_t w_rows_per_cloud; /* 0: one weight for all clouds; else row offset between per-cloud weights */
  const float* bias; int32_t bias_stride;
  int32_t act; float act_alpha;
  const float* res; int64_t ldr;
  float* out_f32;  int64_t ldo32;
  void* out_bf16;  int64_t ldo16;
  double* stats;
  const float* geom;        /* [clouds, valid_rows, 3] fp32 raw sampler state x (not yet scaled by c_in) */
  const float* sigma; int32_t sigma_stride; float sigma_data; /* sigma[cloud*sigma_stride] */
  const float* wx;          /* [n_out, 3] fp32 */
  gecco_anorm anorm;        /* anorm.stats == NULL: `a` is used as it is */
} gecco_gemm_args;

int gecco_gemm(const gecco_gemm_args* args, void* stream);
/* 1 when gecco_gemm accepts args->anorm for this problem shape (m % 256 == 0, m >= 2048, rows_per_cloud % 256 == 0,
 * k % 64 == 0, k <= 384, n_out % 96 == 0), else 0: the caller then applies AdaGN separately (gecco_adagn or
 * gecco_fold_adagn). */
int gecco_gemm_anorm_supported(int32_t m, int32_t rows_per_cloud, int32_t n_out, int32_t k);

/* ------------------------------------------------------------------------
 * Fused point-side MLP with residual (BroadcastingLayer.forward, models/set_transformer.py:165-166;
 * MLP, models/mlp.py:5-39; GaussianActivation, models/activation.py:17-24):
 *   out = res + W2 . g(W1_b . a + b1_b) + b2,   g(z) = (exp(-z^2 / (2 alpha^2)) - 0.7) / 0.28
 * a:  bf16 [m, c] (the bf16 copy of the residual stream), W1_b: bf16 [hidden, c] per cloud
 * (w1_rows_per_cloud = row offset between clouds, 0 = shared), b1_b fp32 [clouds][b1_stride];
 * W2: bf16 [c, hidden], b2 fp32 [c].  The hidden activation stays on chip (TMEM -> shared memory).
 * res / out_f32 (may alias), out_bf16, stats, rows_per_cloud, valid_rows as in gecco_gemm.
 * Supported shapes: c == 384, hidden % 128 == 0, m % 256 == 0, rows_per_cloud % 256 == 0
 * (GECCO_ERR_INVALID otherwise; the engine then runs the two projections through gecco_gemm).
 * With args->anorm (hidden == 768) the CTA-pair kernel of mlp_pair.cu runs: AdaGN on the A operand, the hidden tile of
 * a row block parked in an L2-resident scratch between the two products.
 * ------------------------------------------------------------------------ */
typedef struct gecco_mlp_args {
  const void* a;   int64_t lda;
  const void* w1;  int64_t ldw1;  int32_t w1_rows_per_cloud;
  const float* b1; int32_t b1_stride;
  float act_alpha;
  const void* w2;  int64_t ldw2;
  const float* b2;
  int32_t m, c, hidden;
  int32_t rows_per_cloud, valid_rows;
  const float* res; int64_t ldr;
  float* out_f32;  int64_t ldo32;
  void* out_bf16;  int64_t ldo16;
  double* stats;
  gecco_anorm anorm;  /* anorm.stats != NULL: `a` is the un-normalised bf16 residual-stream copy and AdaGN (mlp_norm,
                       * set_transformer.py:165) is applied to the A operand inside the kernel (w1 / b1 shared by all clouds,
                       * w1_rows_per_cloud == 0); needs `scratch` */
  void* scratch;      /* anorm path: bf16 device scratch of min(m, 128 * #SMs) x hidden elements: the hidden activation of
                       * the row block a CTA is working on (rewritten every row block: L2-resident, never read after the call) */
} gecco_mlp_args;

int gecco_mlp(const gecco_mlp_args* args, void* stream);

/* ------------------------------------------------------------------------
 * Group statistics: stats[cloud][c / group_size][{sum, sum of squares}] += over the
 * first valid_rows rows of each cloud (double accumulators, caller zeroes them).
 * The statistics half of nn.GroupNorm as used by AdaGN (models/normalization.py:21-25,37-38)
 * and GroupNormBNC (models/ray.py:20-30).
 * ------------------------------------------------------------------------ */
int gecco_group_stats(const float* x, int64_t ldx, int32_t clouds, int32_t rows_per_cloud, int32_t valid_rows,
                      int32_t c, int32_t group_size, double* stats, void* stream);

/* AdaGN apply (models/normalization.py:36-44):
 *   y[b,n,c] = scale_b(t)[c] * (x[b,n,c] - mean[b,g]) * rstd[b,g] + bias_b(t)[c]
 * scale(t) = t . scale_w[c,:] + scale_b[c], bias likewise (nn.Linear(ctx_dim, C)).
 * stats are kept at stat_gs-channel granularity; the normalisation group is c/groups
 * channels wide (a multiple of stat_gs).  Padding rows are written as zeros. */
typedef struct gecco_adagn_args {
  const float* x; int64_t ldx;
  const double* stats; int32_t stat_gs;
  const float* t; int32_t t_stride; int32_t ctx_dim;
  const float* scale_w; const float* scale_b; const float* bias_w; const float* bias_b;
  int32_t clouds, rows_per_cloud, valid_rows, c, groups;
  float eps;
  void* out_bf16; int64_t ldo16;
  float* out_f32; int64_t ldo32;
} gecco_adagn_args;
int gecco_adagn(const gecco_adagn_args* args, void* stream);

/* AdaGN (models/normalization.py:36-44) followed by an nn.Linear, folded into per-cloud weights so that the
 * projection reads the un-normalised bf16 residual stream:
 *   w_folded[cloud][o][c] = w[o][c] * a[cloud][c],  bias_folded[cloud][o] = bias[o] + sum_c w[o][c] * s[cloud][c]
 *   a = scale(t) * rstd_g,  s = bias(t) - a * mean_g   (mean / rstd from stats over valid_rows * C/groups elements).
 * Used for kv_proj + the unpool q projection (set_transformer.py:49,112) and mlp.0 (mlp.py:5-39). */
typedef struct gecco_fold_adagn_args {
  const float* w; int64_t ldw;      /* fp32 [n_out, C] */
  const float* bias;                /* [n_out] or NULL */
  int32_t n_out, c;
  const double* stats; int32_t stat_gs; int32_t groups; int32_t valid_rows; float eps;
  const float* t; int32_t t_stride; int32_t ctx_dim;
  const float* scale_w; const float* scale_b; const float* bias_w; const float* bias_b;
  int32_t clouds;
  void* w_folded_bf16; int64_t ldwf; int64_t wf_cloud_stride;   /* elements */
  float* bias_folded; int32_t bias_stride;
} gecco_fold_adagn_args;
int gecco_fold_adagn(const gecco_fold_adagn_args* args, void* stream);

/* GaussianActivation.forward (models/activation.py:17-24) as a stand-alone op on n contiguous floats (16-byte aligned):
 * y = exp(-x^2 / (2 alpha^2)), then (y - 0.7) / 0.28 when normalized != 0.  In the denoiser it is fused into the
 * epilogue of the projection that produces x (gecco_gemm `act`). */
int gecco_gaussian_activation(const float* x, float* y, int64_t n, float alpha, int32_t normalized, void* stream);

/* LinearLift.lift (models/linear_lift.py:21,44) on the EDM-scaled input:
 *   x[b,n,:] = W (c_in(sigma_b) * xin[b,n,:]) + bias, c_in = 1/sqrt(sigma_data^2 + sigma^2)
 * (sigma NULL: c_in = 1) and, when stats != NULL, the statistics of x for the first AdaGN. */
typedef struct gecco_lift_args {
  const float* xin;                 /* [clouds, valid_rows, 3] */
  const float* sigma; int32_t sigma_stride; float sigma_data;
  const float* w; const float* b;   /* [C, 3], [C] */
  int32_t clouds, rows_per_cloud, valid_rows, c;
  float* x; int64_t ldx;            /* [clouds*rows_per_cloud, C] */
  void* x_bf16; int64_t ldxb;       /* optional bf16 copy of x (the operand of the first projections) */
  double* stats; int32_t stat_gs;
} gecco_lift_args;
int gecco_lift(const gecco_lift_args* args, void* stream);

/* Output head fused with the EDM preconditioning and the sampler update.
 *   F = W_out . norm(x) + b_out   norm: 0 none, 1 LayerNorm(C) (models/linear_lift.py:26-29),
 *                                       2 GroupNorm(groups) over points (models/ray.py:56-59)
 *   mode 0: out_f32 = F
 *   mode 1: out_f32 = c_skip*xin + c_out*F                               (diffusion.py:46-57)
 *   mode 2: Euler step   d_cur=(x_hat-D)/t_hat; x_next=x_hat+(t_next-t_hat)d_cur   (diffusion.py:335-336)
 *   mode 3: Heun step    x = x_hat+(t_next-t_hat)(d_cur/2+d'/2) (diffusion.py:346-347), then the churn
 *           of the following step x_hat = x + churn_next*noise_next (diffusion.py:323-325)
 * Sampler state is float64 like the reference; xin_next receives the fp32 input of the next evaluation. */
typedef struct gecco_head_args {
  const float* x; int64_t ldx;
  int32_t clouds, rows_per_cloud, valid_rows, c;
  int32_t norm, groups; const double* stats; int32_t stat_gs; float eps;
  const float* w_out; const float* b_out;
  const float* xin;
  const float* sigma; int32_t sigma_stride; float sigma_data;
  int32_t mode;
  float* out_f32;
  double* x_hat; double* x_next; double* d_cur; float* xin_next; const float* noise_next;
  double t_hat, t_next, churn_next;
} gecco_head_args;
int gecco_head(const gecco_head_args* args, void* stream);

/* Reparametrisations (reparam.py:31-201): kind 0 NoReparam, 1 GaussianReparam, 2 UVLReparam;
 * to_data != 0 is diffusion_to_data, else data_to_diffusion.  in/out are [clouds, points, 3]
 * float (is_double == 0) or double.  mean/sigma are HOST arrays of 3 floats; K is the device
 * [clouds,3,3] fp32 camera matrix (UVL only). */
int gecco_reparam(const void* in, void* out, int32_t is_double, int32_t kind, int32_t to_data,
                  const float* host_mean, const float* host_sigma, float logit_scale, const float* K,
                  int32_t clouds, int32_t points_per_cloud, void* stream);

/* ------------------------------------------------------------------------
 * Projective feature lookup: RayNetwork.extract_image_features (models/ray.py:64-87),
 * i.e. reparam.diffusion_to_data -> kornia project_points -> F.grid_sample(bilinear,
 * zeros padding, align_corners=False) on every pyramid level -> channel concat.
 * The input is the raw sampler state; the EDM input scaling c_in(sigma) is applied inside
 * (sigma NULL: no scaling).  Pyramid levels are bf16 channels-last [clouds, H, W, C]
 * (see gecco_pack_features).  Output rows [cloud*rows_per_cloud + point, sum C] as bf16
 * and/or fp32; optional GroupNorm statistics [clouds][stat_groups][2] of the fp32 result
 * (models/ray.py:53).
 * ------------------------------------------------------------------------ */
#define GECCO_MAX_LEVELS 4
typedef struct gecco_lookup_args {
  const float* xin;                       /* [clouds, points, 3] */
  const float* sigma; int32_t sigma_stride; float sigma_data;
  int32_t reparam;                        /* 0 none, 1 gaussian, 2 uvl */
  float mean[3]; float sigma_r[3]; float logit_scale;
  const float* K;                         /* [clouds, 3, 3] */
  int32_t n_levels;
  const void* level_ptr[GECCO_MAX_LEVELS];
  int32_t level_h[GECCO_MAX_LEVELS], level_w[GECCO_MAX_LEVELS], level_c[GECCO_MAX_LEVELS];
  int32_t clouds, points, rows_per_cloud;
  void* out_bf16; int64_t ldo16;
  float* out_f32; int64_t ldo32;
  double* stats; int32_t stat_groups;
} gecco_lookup_args;
int gecco_lookup(const gecco_lookup_args* args, void* stream);

/* nn.Sequential(GroupNormBNC(groups, c_in, affine=False), nn.Linear(c_in, c_out)) (models/ray.py:52-55)
 * folded into per-cloud weights:  w_folded[cloud][o][c] = w[o][c]*rstd, bias_folded[cloud][o] =
 * bias[o] - sum_c w[o][c]*mean*rstd, with mean/rstd from stats [clouds][groups][2] over `count` elements. */
int gecco_fold_group_norm(const float* w, const float* bias, const double* stats, double count, float eps,
                          int32_t groups, int32_t c_in, int32_t c_out, int32_t clouds, void* w_folded_bf16,
                          int64_t ldw, float* bias_folded, void* stream);

/* Conditioner hand-off: fp32 NCHW feature map (models/feature_pyramid.py:62-73) -> bf16 NHWC. */
int gecco_pack_features(const float* nchw, void* nhwc_bf16, int32_t images, int32_t c, int32_t h, int32_t w,
                        void* stream);

/* ------------------------------------------------------------------------
 * AttentionPool's scaled_dot_product_attention with the learned inducer queries
 * (models/set_transformer.py:57-63).  kv holds the bf16 kv_proj output, K of head h at
 * columns k_off + h*head_dim, V at v_off + h*head_dim ("b n (t h d)" layout, :50-55).
 * q_inducers: bf16 [heads][64][head_dim] = inducers * (head_dim^-0.5 * log2 e).
 * The keys are processed in `splits` ranges; partial is scratch of
 * clouds*heads*splits*64*(head_dim+2) floats.  out: bf16 [clouds*64, heads*head_dim]
 * ("b h i d -> b i (h d)", :63), the operand of out_proj.
 * ------------------------------------------------------------------------ */
typedef struct gecco_pool_args {
  const void* kv; int64_t ld; int32_t k_off, v_off;
  int32_t clouds, rows_per_cloud, valid_rows;
  int32_t heads, head_dim, inducers;
  const void* q_inducers;
  int32_t splits; float* partial;
  void* out_bf16; int64_t ldo;
} gecco_pool_args;
int gecco_pool_attention(const gecco_pool_args* args, void* stream);
/* The same without the final merge of the key splits: *splits_used > 1 means args->partial holds that many (acc, max, sum)
 * partials per (cloud, head, inducer) for gecco_inducer_chain to merge; 1 means args->out_bf16 is final. */
int gecco_pool_attention_partial(const gecco_pool_args* args, int32_t* splits_used, void* stream);

/* Attention core of Broadcast.unpool = nn.MultiheadAttention(query=points, key=value=inducers)
 * (models/set_transformer.py:90,112) between the in- and out-projections: per head
 * softmax(q k^T) v over the 64 inducers.  q: bf16 rows [clouds*rows_per_cloud] with head h at
 * columns h*head_dim, already multiplied by head_dim^-0.5 * log2 e (folded into the q
 * projection); kv: bf16 [clouds*64, *] with k at column h*head_dim and v at v_off + h*head_dim. */
typedef struct gecco_unpool_args {
  const void* q; int64_t ldq;
  const void* kv; int64_t ldkv; int32_t v_off;
  int32_t clouds, rows_per_cloud;
  int32_t heads, head_dim, inducers;
  void* out_bf16; int64_t ldo;
  void* vt_scratch;   /* optional bf16 [clouds * heads * head_dim * inducers] device scratch (v transposed per cloud): when given
                       * and heads == 8, head_dim == 48, rows_per_cloud % 128 == 0 the tcgen05 / TMEM kernel runs, otherwise
                       * (NULL or other shapes) the mma.sync kernel */
  int32_t vt_ready;   /* nonzero: vt_scratch already holds V transposed (written by gecco_inducer_chain) */
} gecco_unpool_args;
int gecco_unpool_attention(const gecco_unpool_args* args, void* stream);

/* The inducer side of Broadcast.forward (models/set_transformer.py:106-112) in one launch:
 *   pooled (or the key-split partials of gecco_pool_attention) -> pool.out_proj -> norm_1 (AdaGN) -> mlp
 *   (Linear, Gaussian activation, Linear) -> norm_2 (AdaGN) -> unpool key | value in-projection (+ V transposed per cloud).
 * A cluster of four CTAs owns two clouds; the AdaGN statistics over (64 inducers, 12 channels) are computed inside the
 * producing accumulator tile.  Shapes: 64 inducers, C = 384, hidden = 768, 8 heads, 32 groups (gecco-torch's only
 * configuration); gecco_inducer_chain returns GECCO_ERR_INVALID for anything else (the engine then runs the stages as
 * separate gecco_gemm / gecco_adagn launches).
 * first_stage 0: the whole chain; 3: only h3 -> k | v (the caller put the cached inducer states, bf16, into h3).
 * Weights are bf16 [n_out, k] row-major (nn.Linear layout); all activation buffers are bf16 [clouds*64, C or hidden]:
 * pooled / hn / h3 [.., C], hh [.., hidden], khv [.., 2C] (k | v); vt: optional bf16 [clouds][C][64]; cache_out: optional
 * fp32 [clouds*64, C] copy of the norm_2 output (the `hs` entry of SetTransformer.forward, :211). */
typedef struct gecco_chain_args {
  int32_t clouds, inducers, c, hidden, heads, groups;
  int32_t first_stage;
  const float* partial; int32_t splits;   /* splits <= 1: pooled is final */
  void* pooled;
  const void *w_pool_out, *w_mlp0, *w_mlp2, *w_kv;
  const float *b_mlp0, *b_mlp2, *b_kv;
  float act_alpha;
  const float* norm[2][4];                /* norm_1 / norm_2: scale.weight, scale.bias, bias.weight, bias.bias, [C] each */
  const float* t; int32_t t_stride; float eps;
  void *hn, *hh, *h3, *khv, *vt;
  float* cache_out;
} gecco_chain_args;
int gecco_inducer_chain(const gecco_chain_args* args, void* stream);

/* ========================================================================
 * Denoiser engine: one handle per (model, device).  This is the entry a maintainer binds in place of
 * Diffusion.forward / EDMPrecond.forward (diffusion.py:233-247, 37-62) and of the body of
 * Diffusion.sample_stochastic / Diffusion.upsample (diffusion.py:271-352, 354-470).
 * ======================================================================== */
#define GECCO_MAX_LAYERS 32

typedef struct gecco_model_desc {
  int32_t kind;          /* 0: LinearLift (models/linear_lift.py), 1: RayNetwork (models/ray.py) */
  int32_t n_layers, feature_dim, num_heads, num_inducers, mlp_hidden;
  int32_t adagn_groups;  /* 32 (models/normalization.py:19) */
  int32_t head_norm;     /* 0 none, 1 LayerNorm (linear_lift.py:26-29), 2 GroupNorm over points (ray.py:56-59) */
  int32_t head_groups;   /* 16 */
  int32_t img_groups;    /* 16 (ray.py:53) */
  int32_t n_levels; int32_t level_c[GECCO_MAX_LEVELS];
  int32_t reparam;       /* reparam of the lookup: 0 none, 1 gaussian, 2 uvl (ray.py:71) */
  float mean[3], sigma[3], logit_scale;
  float sigma_data;      /* EDMPrecond.sigma_data (diffusion.py:31) */
} gecco_model_desc;

/* fp32 device pointers in the reference state_dict schema (SURVEY.md §8b). */
enum gecco_net_weight {
  GECCO_NW_EMBED_W = 0,  /* lift.weight | xyz_embed.weight           [C,3] */
  GECCO_NW_EMBED_B,      /* lift.bias | xyz_embed.bias               [C]   */
  GECCO_NW_IMG_W,        /* img_feature_proj.1.weight (cond)         [C, sum level_c] */
  GECCO_NW_IMG_B,        /* img_feature_proj.1.bias (cond)           [C]   */
  GECCO_NW_OUT_W,        /* lower.1.weight | output_proj.1.weight    [3,C] */
  GECCO_NW_OUT_B,        /* lower.1.bias | output_proj.1.bias        [3]   */
  GECCO_NW_COUNT
};
enum gecco_layer_weight {      /* `layers.{l}.` + ...  (models/set_transformer.py) */
  GECCO_LW_BN = 0,             /* broadcast_norm.{scale.weight, scale.bias, bias.weight, bias.bias}: 4 entries */
  GECCO_LW_INDUCERS = 4,       /* broadcast.pool.inducers          [1,H,I,d] */
  GECCO_LW_POOL_KV_W,          /* broadcast.pool.kv_proj.weight    [2C,C] */
  GECCO_LW_POOL_OUT_W,         /* broadcast.pool.out_proj.weight   [C,C]  */
  GECCO_LW_N1 = 7,             /* broadcast.norm_1.*: 4 entries */
  GECCO_LW_BMLP_W0 = 11,       /* broadcast.mlp.0.weight [hid,C], .0.bias, .1.alpha (scalar), .2.weight [C,hid], .2.bias */
  GECCO_LW_BMLP_B0, GECCO_LW_BMLP_ALPHA, GECCO_LW_BMLP_W2, GECCO_LW_BMLP_B2,
  GECCO_LW_N2 = 16,            /* broadcast.norm_2.*: 4 entries */
  GECCO_LW_UNPOOL_IN_W = 20,   /* broadcast.unpool.in_proj_weight [3C,C], in_proj_bias [3C], out_proj.weight [C,C], out_proj.bias [C] */
  GECCO_LW_UNPOOL_IN_B, GECCO_LW_UNPOOL_OUT_W, GECCO_LW_UNPOOL_OUT_B,
  GECCO_LW_MN = 24,            /* mlp_norm.*: 4 entries */
  GECCO_LW_MLP_W0 = 28,        /* mlp.0.weight, .0.bias, .1.alpha, .2.weight, .2.bias */
  GECCO_LW_MLP_B0, GECCO_LW_MLP_ALPHA, GECCO_LW_MLP_W2, GECCO_LW_MLP_B2,
  GECCO_LW_COUNT = 33
};

typedef struct gecco_engine gecco_engine;

/* Packs the fp32 weights into the kernel layouts (bf16 operands, folded softmax scale).  The fp32 arrays
 * that are used in place (biases, AdaGN linears, embed / head weights) must stay alive and unchanged
 * until gecco_destroy; re-create the handle after a weight update.  Synchronises `stream` once. */
int gecco_create(const gecco_model_desc* desc, const float* const* net_weights /* [GECCO_NW_COUNT] */,
                 const float* const* layer_weights /* [n_layers * GECCO_LW_COUNT] */, void* stream,
                 gecco_engine** out);
int gecco_destroy(gecco_engine* e);
/* Scratch needed by gecco_denoise / gecco_sample for `clouds` clouds of `points` points. */
int64_t gecco_workspace_bytes(const gecco_engine* e, int32_t clouds, int32_t points);

typedef struct gecco_context {          /* conditional models only */
  const void* level_ptr[GECCO_MAX_LEVELS];        /* bf16 NHWC pyramid levels (gecco_pack_features) */
  int32_t level_h[GECCO_MAX_LEVELS], level_w[GECCO_MAX_LEVELS];
  const float* K;                                  /* [clouds,3,3] */
} gecco_context;

/* One denoiser evaluation (Diffusion.forward -> EDMPrecond.forward -> network):
 *   mode 0: out = F(c_in x, ln(sigma)/4)             raw network output
 *   mode 1: out = c_skip x + c_out F                 (diffusion.py:57)
 *   mode 2 / 3: Euler / Heun(+churn) update of the float64 sampler state, see gecco_head_args.
 * cache_in  != NULL: inducer states h [n_layers][clouds][inducers][C] fp32 are used instead of pooling
 *                    (set_transformer.py:106-110, the upsampling fast path);
 * cache_out != NULL: the inducer states of this evaluation are written there (do_cache). */
typedef struct gecco_denoise_args {
  const float* x;                      /* [clouds, points, 3] */
  const float* sigma; int32_t sigma_stride; float sigma_imm; /* sigma[cloud*stride], or sigma_imm when NULL */
  /* network-level call (LinearLift.forward / RayNetwork.forward, mode 0 only): when t_embed != NULL, x is the
   * already scaled geometry and t_embed[cloud*t_stride] the noise embedding; sigma is ignored. */
  const float* t_embed; int32_t t_stride;
  int32_t clouds, points;
  gecco_context ctx;
  const float* cache_in; float* cache_out;
  int32_t mode;
  float* out;
  double* x_hat; double* x_next; double* d_cur; float* xin_next; const float* noise_next;
  double t_hat, t_next, churn_next;
  void* workspace; int64_t workspace_bytes;
} gecco_denoise_args;
int gecco_denoise(gecco_engine* e, const gecco_denoise_args* args, void* stream);

/* The whole stochastic sampler loop (diffusion.py:305-347) on pre-drawn noise: 2*num_steps-1 evaluations with
 * the preconditioning, churn, Euler and Heun arithmetic fused into the head kernel of each evaluation.
 * host_t_steps: float64 [num_steps+1] (Diffusion.t_steps, last = 0); host_gamma: float64 [num_steps]
 * (diffusion.py:318-322).  noise: [num_steps][clouds][points][3] in the reference draw order.
 * x_out: float64 [clouds, points, 3], the diffusion-space result (reparam.diffusion_to_data is applied by the caller). */
typedef struct gecco_sample_args {
  int32_t clouds, points, num_steps;
  const double* host_t_steps; const double* host_gamma; double s_noise;
  const float* latents; const float* noise;
  gecco_context ctx;
  double* x_out;
  void* workspace; int64_t workspace_bytes;
} gecco_sample_args;
int gecco_sample(gecco_engine* e, const gecco_sample_args* args, void* stream);
/* How the last gecco_sample call on this handle ran: 0 eager (graphs off, profiling, or the caller's stream is itself
 * being captured), 1 captured into a CUDA graph and launched, 2 replayed a cached graph, -1 capture failed and the
 * call ran eagerly.  A graph is reused only when every argument (shapes, schedule, all pointers) is identical. */
int gecco_graph_status(const gecco_engine* e);

/* One step of Diffusion.upsample (diffusion.py:427-466): re-noise the seed cloud to t_cur, one full evaluation on it that
 * caches the inducer states, then num_substeps x { churn, cached Euler evaluation, cached Heun evaluation (unless
 * last_step), re-noise (unless the last sub-step or last_step) } on the new points, with the preconditioning and the
 * Euler / Heun arithmetic fused into the head kernel of each cached evaluation and float64 sampler state.
 *   seed_data  [clouds, seed_points, 3] fp32  diffusion-space seed cloud (reparam.data_to_diffusion of the input)
 *   seed_noise [clouds, seed_points, 3] fp32  the step's `randn(data.shape)`
 *   noise      fp32 draws on the new points in the reference order: churn_0, redo_0, churn_1, ..., churn_{S-1}
 *              ([2S-1][clouds, new_points, 3]; last_step: churn_0 .. churn_{S-1}, [S][...])
 *   x          float64 [clouds, new_points, 3]: x_next of the previous step in, x_next of this step out.
 * t_hat = t_cur + gamma t_cur; churn = sqrt(t_hat^2 - t_cur^2) s_noise; redo = sqrt(t_cur^2 - t_next^2). */
typedef struct gecco_upsample_step_args {
  int32_t clouds, seed_points, new_points, num_substeps, last_step;
  double t_cur, t_next, gamma, s_noise;
  const float* seed_data; const float* seed_noise; const float* noise;
  double* x;
  gecco_context ctx;
  void* workspace; int64_t workspace_bytes;
} gecco_upsample_step_args;
int64_t gecco_upsample_workspace_bytes(const gecco_engine* e, int32_t clouds, int32_t seed_points, int32_t new_points);
int gecco_upsample_step(gecco_engine* e, const gecco_upsample_step_args* args, void* stream);

/* ---------------------------------------------------------------------------
 * Training-step tail (BASELINE config 5): torch.optim.Adam (the reference's configure_optimizers, diffusion.py:207-208;
 * defaults betas (0.9, 0.999), eps 1e-8, no weight decay) fused with the weight EMA of ema.py:187-194
 * (ema = decay * ema + (1 - decay) * p_new) over FLAT fp32 buffers of n elements, one launch:
 *   g' = grad_scale * g;  m = b1 m + (1-b1) g';  v = b2 v + (1-b2) g'^2;
 *   p -= lr / (1 - b1^step) * m / (sqrt(v) / sqrt(1 - b2^step) + eps);   ema (may be NULL) updated from the new p.
 * `step` counts from 1.  All buffers 16-byte aligned.  The scalars are doubles so that 1 - beta and the bias corrections
 * are formed exactly like torch forms them from Python floats before rounding to fp32.
 * ------------------------------------------------------------------------ */
int gecco_adam_ema_step(float* p, const float* g, float* m, float* v, float* ema, int64_t n, int64_t step, double lr,
                        double beta1, double beta2, double eps, double grad_scale, double ema_decay, void* stream);

/* ------------------------------------------------------------------------
 * Element-wise kernels of the training step's autograd functions (gecco_b200/training.py), one HBM-bound pass each:
 *   GaussianActivation (models/activation.py:17-24), forward and backward, with alpha as a DEVICE scalar (no host
 *   read-back: the step is captured as a CUDA graph); the backward writes gecco_train_gauss_act_bwd_parts(n) partial
 *   sums of dalpha (one per block; the caller adds them up in a fixed order -- deterministic, no atomics);
 *   the two kernels of AdaGN / GroupNorm (models/normalization.py:36-44, models/ray.py:20-30) around gecco_group_stats:
 *     affine : out[b,n,c] = p[b,c] * u[b,n,c] (+ q[b,c] * w[b,n,c]) + r[b,c]   (w, q both NULL or both given)
 *              forward y = gamma * xhat + beta with (u = x) and the input gradient with (u = dy, w = x);
 *     colsum2: out[b,part,c,0] = partial sum_n dy[b,n,c], out[b,part,c,1] = partial sum_n dy[b,n,c] * x[b,n,c] for the
 *              gecco_train_colsum2_parts(rows_per_cloud, c) row partitions of a cloud (the caller sums over `part`).
 * All tensors contiguous fp32 [clouds, rows_per_cloud, c], c a multiple of 4 (<= 1024), 16-byte aligned.
 * ------------------------------------------------------------------------ */
int gecco_train_gauss_act_fwd(const float* x, const float* alpha, float* y, int64_t n, int32_t normalized, void* stream);
int64_t gecco_train_gauss_act_bwd_parts(int64_t n);
int gecco_train_gauss_act_bwd(const float* x, const float* dy, const float* alpha, float* dx, float* dalpha, int64_t n,
                              int32_t normalized, void* stream);
int gecco_train_affine(const float* u, const float* w, const float* p, const float* q, const float* r, float* out,
                       int32_t clouds, int32_t rows_per_cloud, int32_t c, void* stream);
int32_t gecco_train_colsum2_parts(int32_t rows_per_cloud, int32_t c);
int gecco_train_colsum2(const float* dy, const float* x, float* out, int32_t clouds, int32_t rows_per_cloud, int32_t c,
                        void* stream);

/* ------------------------------------------------------------------------
 * Chamfer distance between point clouds, the distance under the 1-NNA / MMD / COV sample-quality metrics
 * (gecco_b200/metrics.py; PointFlow's compute_all_metrics protocol; gecco-jax metrics.py has the same role):
 *   CD(X, Y) = mean_{x in X} min_{y in Y} |x - y|^2 + mean_{y in Y} min_{x in X} |x - y|^2
 * (squared Euclidean distances, means not sums, no normalisation of the clouds).
 * a: fp32 [ma, na, 3] contiguous, b: fp32 [mb, nb, 3] contiguous; na, nb >= 1, the smaller of the two at most 32768.
 * mode GECCO_CHAMFER_ALL   : out [ma, mb], out[i][j] = CD(a[i], b[j]);
 *      GECCO_CHAMFER_PAIRED: out [ma],     out[i] = CD(a[i], b[i]), ma == mb (bitwise equal to the ALL diagonal);
 *      GECCO_CHAMFER_SELF  : out [ma, ma], CD(a[i], a[j]); b is NULL or a; each pair i < j is computed once and written to
 *                            both halves (exactly symmetric), the diagonal is exactly 0.
 * One block per cloud pair, both directions in one pass; results are bitwise deterministic.  Non-finite points are not
 * detected here (the minima would silently skip NaN): the caller checks its input.
 * ------------------------------------------------------------------------ */
#define GECCO_CHAMFER_ALL 0
#define GECCO_CHAMFER_PAIRED 1
#define GECCO_CHAMFER_SELF 2
typedef struct gecco_chamfer_args {
  const float* a; int32_t ma, na;
  const float* b; int32_t mb, nb;
  int32_t mode;
  float* out;
} gecco_chamfer_args;
int gecco_chamfer(const gecco_chamfer_args* args, void* stream);

/* Per-kernel-class device timing of the engine (tracing aid; the reference has none, SURVEY.md §5).  Between
 * start and stop every engine launch on this thread is bracketed by CUDA events on its stream; stop synchronises
 * the device and returns, per class, the launch count, summed device time and the algorithmic FLOPs / bytes. */
typedef struct gecco_profile_entry {
  char name[32];
  int64_t launches;
  double ms, flops, bytes;
} gecco_profile_entry;
int gecco_profile_start(void);
int gecco_profile_stop(gecco_profile_entry* out, int32_t capacity, int32_t* count);

/* Number of kernel launches the library has issued on this thread since the last call (bench bookkeeping). */
int64_t gecco_launch_count(int32_t reset);

#ifdef __cplusplus
}
#endif
#endif /* GECCO_B200_H */
