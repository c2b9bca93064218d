// Denoiser engine: sequences the kernels of one EDM-preconditioned SetTransformer evaluation
// (Diffusion.forward, diffusion.py:233-247) and the stochastic sampler loop around it
// (Diffusion.sample_stochastic, diffusion.py:305-347) on one stream.  No host synchronisation, no
// allocation after gecco_create: everything is CUDA-graph capturable.
#include "kernels.cuh"
#include "ptx.cuh"

#include <math.h>
#include <new>
#include <stdlib.h>
#include <string.h>
#include <vector>

// ---------------------------------------------------------------------------------------------
// Per-kernel-class device timing (gecco_profile_start / gecco_profile_stop): when enabled, every launch of the
// engine is bracketed by CUDA events on the launching stream and attributed to a class together with its
// algorithmic FLOPs and bytes.  Off by default (no events, no overhead).
namespace gecco {
namespace {
enum KClass {
  K_PREP = 0, K_LIFT, K_LOOKUP, K_FOLD_GN, K_GEMM_IMG, K_FOLD_ADAGN, K_GEMM_KVQ, K_POOL_ATTN, K_INDUCER_CHAIN,
  K_UNPOOL_ATTN, K_GEMM_UNPOOL_OUT, K_GEMM_MLP0, K_GEMM_MLP2, K_MLP_FUSED, K_HEAD, K_MISC, K_COUNT
};
const char* const kClassNames[K_COUNT] = {
    "prep", "lift", "lookup", "fold_group_norm", "gemm_img_proj", "fold_adagn", "gemm_kv_q", "pool_attention",
    "inducer_chain", "unpool_attention", "gemm_unpool_out", "gemm_mlp_up_act", "gemm_mlp_down", "mlp_fused",
    "head_edm_step", "misc"};
struct Profiler {
  bool on = false;
  std::vector<cudaEvent_t> pool;
  size_t used = 0;
  struct Rec { int cls; size_t ev; double flops, bytes; };
  std::vector<Rec> recs;
  cudaEvent_t take() {
    if (used == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[used++];
  }
};
thread_local Profiler g_prof;
inline void prof_begin(int cls, double flops, double bytes, cudaStream_t s) {
  if (!g_prof.on) return;
  g_prof.recs.push_back({cls, g_prof.used, flops, bytes});
  cudaEventRecord(g_prof.take(), s);
  g_prof.take();
}
inline void prof_end(cudaStream_t s) {
  if (!g_prof.on) return;
  cudaEventRecord(g_prof.pool[g_prof.recs.back().ev + 1], s);
}
}  // namespace
}  // namespace gecco

struct gecco_engine {
  gecco_model_desc d;
  int device;
  // fp32 tensors used in place (owned by the caller)
  const float* net[GECCO_NW_COUNT];
  std::vector<const float*> lw;  // [n_layers * GECCO_LW_COUNT]
  // packed (owned)
  struct Layer {
    __nv_bfloat16 *pool_out_w, *bmlp_w0, *bmlp_w2, *kv_w, *out_w, *mlp_w2, *q_ind;
    // bf16 copies of the projections that follow an AdaGN, for the GEMM that normalises its A operand itself
    // (gecco_anorm): [kv_proj.weight ; qscale * in_proj_weight[0:C]] and mlp.0.weight
    __nv_bfloat16 *wcat16, *mlp_w0;
    // fp32 sources of the AdaGN-folded projections: [kv_proj.weight ; qscale * in_proj_weight[0:C]] and its bias
    float *wcat, *bcat;
    float bmlp_alpha, mlp_alpha;
  };
  std::vector<Layer> layers;
  float* img_bias;  // img_feature_proj.1.bias + xyz_embed.bias (cond)
  void* arena;      // one allocation holding all packed tensors
  size_t arena_bytes;
  // CUDA graphs of whole sampler loops (gecco_sample): captured once per distinct argument set, replayed afterwards.
  // Captured and replayed on the engine's own stream, forked from / joined to the caller's stream with events, so that
  // the legacy default stream (which cannot be captured) works too.
  struct SampleGraph {
    std::vector<unsigned char> key;
    cudaGraphExec_t exec;
    long long launches;  // kernel launches one replay performs
    unsigned long long stamp;
  };
  std::vector<SampleGraph> graphs;
  unsigned long long graph_clock = 0;
  cudaStream_t gstream = nullptr;
  cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
  int last_graph_status = 0;  // 0: eager, 1: captured this call, 2: replayed, <0: capture failed (ran eagerly)
};

namespace gecco {

namespace {

__global__ void pack_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, long long n, float scale) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = __float2bfloat16(src[i] * scale);
}
__global__ void scale_add_f32_kernel(const float* __restrict__ a, const float* __restrict__ b, float* __restrict__ dst,
                                     int n, float scale) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = a[i] * scale + (b ? b[i] : 0.f);
}

// Per evaluation: zero the statistics accumulators, materialise sigma per cloud and c_noise = ln(sigma)/4
// (diffusion.py:51).
// Network-level calls pass the embedding directly (t_embed) and an input that is already scaled: sigma_eff = 0
// makes every c_in(sigma) in the downstream kernels equal to 1 / sigma_data, which the engine cancels by
// running them with sigma_data = 1.
__global__ void prep_kernel(double* __restrict__ stats, long long n_stats, const float* __restrict__ sigma, int stride,
                            float sigma_imm, const float* __restrict__ t_embed, int t_stride, int clouds,
                            float* __restrict__ sigma_eff, float* __restrict__ c_noise) {
  pdl_wait();  // programmatic dependent launch: the predecessor (the previous evaluation's head) has completed
  pdl_launch_dependents();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (long long j = i; j < n_stats; j += (long long)gridDim.x * blockDim.x) stats[j] = 0.0;
  if (i < clouds) {
    if (t_embed != nullptr) {
      sigma_eff[i] = 0.f;
      c_noise[i] = t_embed[(long long)i * t_stride];
    } else {
      const float s = sigma ? sigma[(long long)i * stride] : sigma_imm;
      sigma_eff[i] = s;
      c_noise[i] = logf(s) / 4.0f;
    }
  }
}

__global__ void copy_f64_kernel(const double* __restrict__ src, double* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

inline size_t align_up(size_t x, size_t a = 256) { return (x + a - 1) / a * a; }

// Bump allocator over the caller's workspace.
struct Carver {
  uint8_t* base;
  size_t off = 0;
  template <typename T>
  T* take(size_t count) {
    T* p = reinterpret_cast<T*>(base + off);
    off = align_up(off + count * sizeof(T));
    return p;
  }
};

struct Workspace {
  int Np, rows, irows, splits;
  float* x;            // [rows, C] residual stream (fp32)
  __nv_bfloat16* xb;   // [rows, C] bf16 copy of the residual stream: the operand of the AdaGN-folded projections
  __nv_bfloat16* y;    // [rows, C] unpool attention output
  __nv_bfloat16* big;  // [rows, max(3C, hidden, sum level_c)] k|v|q | mlp hidden | looked-up image features
  int wide;
  __nv_bfloat16 *pooled, *hn, *hh, *h3, *khv, *vt;
  float *h, *h2, *partial;
  double* stats;
  long long n_stats;
  float *sigma_eff, *c_noise;
  __nv_bfloat16* wfold;
  float* bfold;
  double *x_hat, *x_next, *d_cur;
  float *xin_a, *xin_b;
  size_t bytes;
};

int pool_splits(int clouds, int heads, int n_tiles) {
  int s = ceil_div(8 * 148, clouds * heads);
  if (s < 1) s = 1;
  if (s > n_tiles) s = n_tiles;
  return s;
}

Workspace carve(const gecco_engine* e, int clouds, int points, void* base) {
  const gecco_model_desc& d = e->d;
  Workspace w;
  const int C = d.feature_dim, I = d.num_inducers, hid = d.mlp_hidden;
  int ctx = 0;
  for (int l = 0; l < d.n_levels; ++l) ctx += d.level_c[l];
  w.Np = ceil_div(points, 128) * 128;
  w.rows = clouds * w.Np;
  w.irows = clouds * I;
  // the mma.sync pool core runs one CTA per 64 inducers of each split
  w.splits = pool_splits(clouds, d.num_heads * (I / 64), ceil_div(points, 64));
  int wide = 3 * C;
  if (hid > wide) wide = hid;
  if (ctx > wide) wide = ctx;
  w.wide = wide;
  Carver c{static_cast<uint8_t*>(base)};
  w.x = c.take<float>((size_t)w.rows * C);
  w.xb = c.take<__nv_bfloat16>((size_t)w.rows * C);
  w.y = c.take<__nv_bfloat16>((size_t)w.rows * C);
  w.big = c.take<__nv_bfloat16>((size_t)w.rows * wide);
  w.pooled = c.take<__nv_bfloat16>((size_t)w.irows * C);
  w.hn = c.take<__nv_bfloat16>((size_t)w.irows * C);
  w.hh = c.take<__nv_bfloat16>((size_t)w.irows * hid);
  w.h3 = c.take<__nv_bfloat16>((size_t)w.irows * C);
  w.khv = c.take<__nv_bfloat16>((size_t)w.irows * 2 * C);
  w.vt = c.take<__nv_bfloat16>((size_t)w.irows * C);  // v transposed per cloud (tcgen05 unpool attention)
  w.h = c.take<float>((size_t)w.irows * C);
  w.h2 = c.take<float>((size_t)w.irows * C);
  w.partial = c.take<float>((size_t)clouds * d.num_heads * w.splits * I * (C / d.num_heads + 2));
  // statistics at the AdaGN group width (C / adagn_groups channels: one sum pair per group): per layer {broadcast_norm,
  // norm_1, norm_2, mlp_norm}, plus the head norm, plus the image-feature GroupNorm
  const int sg = d.adagn_groups;
  w.n_stats = (long long)clouds * ((4LL * d.n_layers + 1) * sg * 2 + (d.kind == 1 ? d.img_groups * 2 : 0));
  w.stats = c.take<double>((size_t)w.n_stats);
  w.sigma_eff = c.take<float>(clouds);
  w.c_noise = c.take<float>(clouds);
  {
    size_t wf = (size_t)3 * C * C;  // [k|v|q] projections folded with broadcast_norm
    if ((size_t)hid * C > wf) wf = (size_t)hid * C;  // mlp.0 folded with mlp_norm
    if ((size_t)C * ctx > wf) wf = (size_t)C * ctx;  // img_feature_proj folded with its GroupNorm
    w.wfold = c.take<__nv_bfloat16>((size_t)clouds * wf);
    w.bfold = c.take<float>((size_t)clouds * (3 * C > hid ? 3 * C : hid));
  }
  const size_t n3 = (size_t)clouds * points * 3;
  w.x_hat = c.take<double>(n3);
  w.x_next = c.take<double>(n3);
  w.d_cur = c.take<double>(n3);
  w.xin_a = c.take<float>(n3);
  w.xin_b = c.take<float>(n3);
  w.bytes = c.off;
  return w;
}

gecco_gemm_args gemm_base(const void* a, long long lda, const void* wgt, long long ldw, int m, int n, int k,
                          int rows_per_cloud, int valid_rows) {
  gecco_gemm_args g = {};
  g.a = a; g.lda = lda; g.w = wgt; g.ldw = ldw;
  g.m = m; g.n_out = n; g.k = k;
  g.rows_per_cloud = rows_per_cloud; g.valid_rows = valid_rows;
  g.sigma_data = 1.f;
  return g;
}

gecco_adagn_args adagn_base(const gecco_engine* e, const float* const* nw /* 4 pointers */, const float* x, const double* stats,
                            const float* t, int clouds, int rows_per_cloud, int valid_rows) {
  gecco_adagn_args a = {};
  const int C = e->d.feature_dim;
  a.x = x; a.ldx = C;
  a.stats = stats; a.stat_gs = C / e->d.adagn_groups;
  a.t = t; a.t_stride = 1; a.ctx_dim = 1;
  a.scale_w = nw[0]; a.scale_b = nw[1]; a.bias_w = nw[2]; a.bias_b = nw[3];
  a.clouds = clouds; a.rows_per_cloud = rows_per_cloud; a.valid_rows = valid_rows; a.c = C;
  a.groups = e->d.adagn_groups;
  a.eps = 1e-5f;
  return a;
}

gecco_fold_adagn_args fold_base(const gecco_engine* e, const float* const* nw /* 4 pointers */, const double* stats,
                                const float* t, int clouds, int valid_rows) {
  gecco_fold_adagn_args a = {};
  a.c = e->d.feature_dim;
  a.stats = stats; a.stat_gs = a.c / e->d.adagn_groups; a.groups = e->d.adagn_groups; a.valid_rows = valid_rows;
  a.eps = 1e-5f;
  a.t = t; a.t_stride = 1; a.ctx_dim = 1;
  a.scale_w = nw[0]; a.scale_b = nw[1]; a.bias_w = nw[2]; a.bias_b = nw[3];
  a.clouds = clouds;
  return a;
}

// gecco_set_option("anorm", 0) keeps the AdaGN -> per-cloud weight fold path everywhere (A/B measurements, tests of the
// fold path at shapes where the A-operand transform would otherwise be taken).
// (Measured and dropped: reading the fp32 stream instead of its bf16 copy -- through a TMA staging ring or straight from
// global memory in the normalising warps -- saves the producers' bf16 write but starves the resident-tile pipeline: the
// k|v|q projection went from 143 to 170-250 us.)
int g_anorm = 1;
// gecco_set_option("chain", 0): the inducer side as separate GEMM / AdaGN launches (A/B measurements, tests)
int g_chain = 1;
// gecco_set_option("mlp_pair", 0): the point-side MLP as two GEMMs with the hidden tensor in HBM
int g_mlp_pair = 1;

#define TRY(expr)            \
  do {                       \
    int rc__ = (expr);       \
    if (rc__ != 0) return rc__; \
  } while (0)

#define TRYP(cls, flops, bytes, expr)   \
  do {                                 \
    prof_begin(cls, flops, bytes, s);  \
    int rc__ = (expr);                 \
    prof_end(s);                       \
    if (rc__ != 0) return rc__;        \
  } while (0)

// Key / value projections (and V^T) of the cached inducer states, per layer.  They depend on the cache only, so the
// upsampling step computes them ONCE in its caching evaluation (mode 1) and its 2 * num_substeps cached evaluations read
// them (mode 2) instead of re-packing the cache and re-projecting it in every layer of every evaluation.
struct KvCache {
  __nv_bfloat16* khv;  // [layers][clouds * I, 2 C]
  __nv_bfloat16* vt;   // [layers][clouds * C, I]
  int mode;            // 1 write, 2 read
};

// One evaluation.  `xin` is the raw (un-scaled) [clouds, points, 3] input; the head arguments select what is
// produced (see gecco_head_args modes).
int run_eval(gecco_engine* e, const Workspace& w, const float* xin, const float* sigma, int sigma_stride, float sigma_imm,
             const float* t_embed, int t_stride, int clouds, int points, const gecco_context& ctx, const float* cache_in, float* cache_out,
             gecco_head_args head, cudaStream_t s, const KvCache* kvc = nullptr) {
  const gecco_model_desc& d = e->d;
  const int C = d.feature_dim, I = d.num_inducers, H = d.num_heads, hid = d.mlp_hidden, hd = C / H;
  const int sg = d.adagn_groups, Np = w.Np, rows = w.rows, irows = w.irows;
  const int act = mlp_act_of(d.mlp_act);  // every MLP's hidden activation, in the epilogue of its first projection
  const long long per_norm = (long long)clouds * sg * 2;
  const float sigma_data = t_embed ? 1.f : d.sigma_data;
  // algorithmic work per launch (profiling only)
  const double Mv = (double)clouds * points, Mi = (double)irows, Cd = C, Hd = hid;
  auto stat = [&](int layer, int which) { return w.stats + ((long long)layer * 4 + which) * per_norm; };
  double* head_stats = w.stats + 4LL * d.n_layers * per_norm;
  double* img_stats = head_stats + per_norm;
  // AdaGN on the point side: normalised inside the consuming GEMM (A-operand transform of the CTA-pair kernel) where
  // the shape allows, else folded into per-cloud weights (fold_adagn + bf16 copy xb of the residual stream).
  const bool an = g_anorm && gemm_anorm_supported(rows, Np, C, C) && gemm_anorm_supported(rows, Np, 3 * C, C) &&
                  gemm_anorm_supported(rows, Np, hid, C);
  __nv_bfloat16* const xb_out = w.xb;  // bf16 copy of the residual stream: the (un-normalised) operand of both paths
  auto set_anorm = [&](gecco_gemm_args& g, const float* const* nw, const double* st) {
    g.anorm.stats = st; g.anorm.stat_gs = C / sg; g.anorm.groups = sg; g.anorm.eps = 1e-5f;
    g.anorm.t = w.c_noise; g.anorm.t_stride = 1;
    g.anorm.scale_w = nw[0]; g.anorm.scale_b = nw[1]; g.anorm.bias_w = nw[2]; g.anorm.bias_b = nw[3];
  };

  {
    const int threads = 256;
    long long need = w.n_stats > clouds ? w.n_stats : clouds;
    int blocks = (int)((need + threads - 1) / threads);
    if (blocks > 1024) blocks = 1024;
    if ((long long)blocks * threads < clouds) blocks = ceil_div(clouds, threads);
    prof_begin(K_PREP, 0, 8.0 * w.n_stats, s);
    launch_small(prep_kernel, dim3(blocks), dim3(threads), 0, s, w.stats, w.n_stats, sigma, sigma_stride, sigma_imm, t_embed, t_stride,
                 clouds, w.sigma_eff, w.c_noise);
    prof_end(s);
    GECCO_CHECK_LAUNCH("prep_kernel");
  }

  // ---------------------------------------------------------------- input embedding
  // Both paths write the fp32 residual stream x, its bf16 copy xb and the statistics of the first AdaGN.
  if (d.kind == 0) {  // LinearLift.lift (models/linear_lift.py:44)
    gecco_lift_args a = {};
    a.xin = xin; a.sigma = w.sigma_eff; a.sigma_stride = 1; a.sigma_data = sigma_data;
    a.w = e->net[GECCO_NW_EMBED_W]; a.b = e->net[GECCO_NW_EMBED_B];
    a.clouds = clouds; a.rows_per_cloud = Np; a.valid_rows = points; a.c = C;
    a.x = w.x; a.ldx = C;
    a.x_bf16 = xb_out; a.ldxb = C;
    a.stats = stat(0, 0); a.stat_gs = C / sg;
    TRYP(K_LIFT, 6 * Mv * Cd, Mv * (Cd * 6 + 12), launch_lift(a, s));
  } else {  // RayNetwork: xyz_embed + img_feature_proj(lookup) (models/ray.py:99-113)
    int ctot = 0;
    gecco_lookup_args a = {};
    a.xin = xin; a.sigma = w.sigma_eff; a.sigma_stride = 1; a.sigma_data = sigma_data;
    a.reparam = d.reparam;
    for (int j = 0; j < 3; ++j) { a.mean[j] = d.mean[j]; a.sigma_r[j] = d.sigma[j]; }
    a.logit_scale = d.logit_scale;
    a.K = ctx.K;
    a.n_levels = d.n_levels;
    for (int l = 0; l < d.n_levels; ++l) {
      a.level_ptr[l] = ctx.level_ptr[l]; a.level_h[l] = ctx.level_h[l]; a.level_w[l] = ctx.level_w[l];
      a.level_c[l] = d.level_c[l];
      ctot += d.level_c[l];
    }
    a.clouds = clouds; a.points = points; a.rows_per_cloud = Np;
    a.out_bf16 = w.big; a.ldo16 = ctot;
    a.stats = img_stats; a.stat_groups = d.img_groups;
    double pyr = 0;
    for (int l = 0; l < d.n_levels; ++l) pyr += 2.0 * clouds * ctx.level_h[l] * ctx.level_w[l] * d.level_c[l];
    TRYP(K_LOOKUP, 8 * Mv * ctot, pyr + Mv * (ctot * 2.0 + 12), launch_lookup(a, s));
    TRYP(K_FOLD_GN, 2.0 * clouds * Cd * ctot, Cd * ctot * (4.0 + 2.0 * clouds),
         launch_fold_gn(e->net[GECCO_NW_IMG_W], e->img_bias, img_stats, (double)points * (ctot / d.img_groups), 1e-5f,
                        d.img_groups, ctot, C, clouds, w.wfold, ctot, w.bfold, s));
    gecco_gemm_args g = gemm_base(w.big, ctot, w.wfold, ctot, rows, C, ctot, Np, points);
    g.w_rows_per_cloud = C;
    g.bias = w.bfold; g.bias_stride = C;
    g.geom = xin; g.sigma = w.sigma_eff; g.sigma_stride = 1; g.sigma_data = sigma_data;
    g.wx = e->net[GECCO_NW_EMBED_W];
    g.out_f32 = w.x; g.ldo32 = C;
    g.out_bf16 = xb_out; g.ldo16 = C;
    g.stats = stat(0, 0); g.stat_gs = C / sg;
    TRYP(K_GEMM_IMG, 2 * Mv * Cd * ctot + 6 * Mv * Cd, Mv * (ctot * 2.0 + Cd * 6) + 2.0 * clouds * Cd * ctot, launch_gemm(g, s));
  }

  // ---------------------------------------------------------------- SetTransformer (models/set_transformer.py:198-216)
  const int C3 = 3 * C;
  for (int l = 0; l < d.n_layers; ++l) {
    const gecco_engine::Layer& L = e->layers[l];
    const float* const* lw = e->lw.data() + (size_t)l * GECCO_LW_COUNT;
    // y = AdaGN_bn(x, t) (:162) is never materialised: it is folded into the per-cloud weights of its two consumers,
    // AttentionPool.kv_proj (:49) and the unpool query projection (:112), which then read xb directly.
    const bool pooling = cache_in == nullptr;
    const int r0 = pooling ? 0 : 2 * C;  // the cached pass only needs the q rows
    if (an) {
      gecco_gemm_args g = gemm_base(w.xb, C, L.wcat16 + (size_t)r0 * C, C, rows, C3 - r0, C, Np, points);
      set_anorm(g, lw + GECCO_LW_BN, stat(l, 0));
      g.bias = L.bcat + r0; g.bias_stride = 0;
      g.out_bf16 = w.big + r0; g.ldo16 = C3;
      TRYP(K_GEMM_KVQ, 2 * Mv * Cd * (C3 - r0), Mv * (Cd * 2 + (C3 - r0) * 2.0) + 2.0 * (C3 - r0) * Cd, launch_gemm(g, s));
    } else {
      gecco_fold_adagn_args f = fold_base(e, lw + GECCO_LW_BN, stat(l, 0), w.c_noise, clouds, points);
      f.w = L.wcat + (size_t)r0 * C; f.ldw = C; f.bias = L.bcat + r0; f.n_out = C3 - r0;
      f.w_folded_bf16 = w.wfold + (size_t)r0 * C; f.ldwf = C; f.wf_cloud_stride = (long long)C3 * C;
      f.bias_folded = w.bfold + r0; f.bias_stride = C3;
      TRYP(K_FOLD_ADAGN, 2.0 * clouds * (C3 - r0) * Cd, (C3 - r0) * Cd * (4.0 + 2.0 * clouds), launch_fold_adagn(f, s));
      gecco_gemm_args g = gemm_base(w.xb, C, w.wfold + (size_t)r0 * C, C, rows, C3 - r0, C, Np, points);
      g.w_rows_per_cloud = C3;
      g.bias = w.bfold + r0; g.bias_stride = C3;
      g.out_bf16 = w.big + r0; g.ldo16 = C3;
      TRYP(K_GEMM_KVQ, 2 * Mv * Cd * (C3 - r0), Mv * (Cd * 2 + (C3 - r0) * 2.0) + 2.0 * clouds * (C3 - r0) * Cd, launch_gemm(g, s));
    }
    gecco_pool_args pool = {};
    pool.kv = w.big; pool.ld = C3; pool.k_off = 0; pool.v_off = C;
    pool.clouds = clouds; pool.rows_per_cloud = Np; pool.valid_rows = points;
    pool.heads = H; pool.head_dim = hd; pool.inducers = I;
    pool.q_inducers = L.q_ind;
    pool.splits = w.splits; pool.partial = w.partial;
    pool.out_bf16 = w.pooled; pool.ldo = C;
    // the inducer side in one cluster kernel (inducer_chain.cu) where the shape allows
    gecco_chain_args ch = {};
    ch.clouds = clouds; ch.inducers = I; ch.c = C; ch.hidden = hid; ch.heads = H; ch.groups = sg;
    ch.pooled = w.pooled;
    ch.w_pool_out = L.pool_out_w; ch.w_mlp0 = L.bmlp_w0; ch.w_mlp2 = L.bmlp_w2; ch.w_kv = L.kv_w;
    ch.b_mlp0 = lw[GECCO_LW_BMLP_B0]; ch.b_mlp2 = lw[GECCO_LW_BMLP_B2]; ch.b_kv = lw[GECCO_LW_UNPOOL_IN_B] + C;
    ch.act_alpha = L.bmlp_alpha; ch.act = act;
    for (int i = 0; i < 4; ++i) { ch.norm[0][i] = lw[GECCO_LW_N1 + i]; ch.norm[1][i] = lw[GECCO_LW_N2 + i]; }
    ch.t = w.c_noise; ch.t_stride = 1; ch.eps = 1e-5f;
    // key / value projections of this layer's inducer states: the workspace buffers, or the per-layer slots of the
    // upsampling step's cache
    __nv_bfloat16* khv_l = kvc ? kvc->khv + (size_t)l * irows * 2 * C : w.khv;
    __nv_bfloat16* vt_l = kvc ? kvc->vt + (size_t)l * irows * C : w.vt;
    ch.hn = w.hn; ch.hh = w.hh; ch.h3 = w.h3; ch.khv = khv_l; ch.vt = vt_l;
    const bool chain = g_chain && inducer_chain_supported(ch);
    bool kv_done = false;
    if (pooling && chain) {
      int nsplit = 1;
      // few key splits are merged by the chain kernel itself; many (small batches: up to one split per 128-point tile) by
      // the wide merge kernel, which spreads them over the whole machine
      if (pool.splits <= 4) {
        TRYP(K_POOL_ATTN, 4 * Mv * I * Cd, Mv * Cd * 4 + Mi * Cd * 2, launch_pool_attention_partial(pool, s, &nsplit));
      } else {
        TRYP(K_POOL_ATTN, 4 * Mv * I * Cd, Mv * Cd * 4 + Mi * Cd * 2, launch_pool_attention(pool, s));
      }
      ch.first_stage = 0;
      ch.partial = w.partial; ch.splits = nsplit;
      if (cache_out != nullptr) ch.cache_out = cache_out + (size_t)l * irows * C;
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd * (2 * Cd + 2 * Hd) + 2 * Mi * Cd * 2 * Cd, Mi * Cd * 8 + 2 * (2 * Cd * Cd + 2 * Cd * Hd + 2 * Cd * Cd),
           launch_inducer_chain(ch, s));
      kv_done = true;
    } else if (pooling) {
      // AttentionPool (:47-65)
      TRYP(K_POOL_ATTN, 4 * Mv * I * Cd, Mv * Cd * 4 + Mi * Cd * 2, launch_pool_attention(pool, s));
      gecco_gemm_args g = gemm_base(w.pooled, C, L.pool_out_w, C, irows, C, C, I, I);
      g.out_f32 = w.h; g.ldo32 = C; g.stats = stat(l, 1); g.stat_gs = C / sg;
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd * Cd, Mi * Cd * 6 + 2 * Cd * Cd, launch_gemm(g, s));
      // h = norm_2(mlp(norm_1(h)))  (:108-110)
      gecco_adagn_args a = adagn_base(e, lw + GECCO_LW_N1, w.h, stat(l, 1), w.c_noise, clouds, I, I);
      a.out_bf16 = w.hn; a.ldo16 = C;
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd, Mi * Cd * 6, launch_adagn(a, s));
      g = gemm_base(w.hn, C, L.bmlp_w0, C, irows, hid, C, I, I);
      g.bias = lw[GECCO_LW_BMLP_B0]; g.act = act; g.act_alpha = L.bmlp_alpha;
      g.out_bf16 = w.hh; g.ldo16 = hid;
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd * Hd, Mi * (Cd + Hd) * 2 + 2 * Cd * Hd, launch_gemm(g, s));
      g = gemm_base(w.hh, hid, L.bmlp_w2, hid, irows, C, hid, I, I);
      g.bias = lw[GECCO_LW_BMLP_B2];
      g.out_f32 = w.h2; g.ldo32 = C; g.stats = stat(l, 2); g.stat_gs = C / sg;
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd * Hd, Mi * (Hd * 2 + Cd * 4) + 2 * Cd * Hd, launch_gemm(g, s));
      a = adagn_base(e, lw + GECCO_LW_N2, w.h2, stat(l, 2), w.c_noise, clouds, I, I);
      a.out_bf16 = w.h3; a.ldo16 = C;
      if (cache_out != nullptr) { a.out_f32 = cache_out + (size_t)l * irows * C; a.ldo32 = C; }
      TRYP(K_INDUCER_CHAIN, 2 * Mi * Cd, Mi * Cd * 6, launch_adagn(a, s));
    } else if (kvc != nullptr && kvc->mode == 2) {
      kv_done = true;  // projected once by the caching evaluation of this noise level
    } else {
      const long long n = (long long)irows * C;
      prof_begin(K_INDUCER_CHAIN, 0, Mi * Cd * 6, s);
      pack_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(cache_in + (size_t)l * irows * C, w.h3, n, 1.0f);
      prof_end(s);
      GECCO_CHECK_LAUNCH("pack_bf16_kernel(cache)");
      if (chain) {
        ch.first_stage = 3;
        TRYP(K_INDUCER_CHAIN, 4 * Mi * Cd * Cd, Mi * Cd * 6 + 4 * Cd * Cd, launch_inducer_chain(ch, s));
        kv_done = true;
      }
    }
    // unpool = nn.MultiheadAttention(query=y, key=value=h)  (:112)
    {
      gecco_gemm_args g;
      if (!kv_done) {
        g = gemm_base(w.h3, C, L.kv_w, C, irows, 2 * C, C, I, I);
        g.bias = lw[GECCO_LW_UNPOOL_IN_B] + C;
        g.out_bf16 = khv_l; g.ldo16 = 2 * C;
        TRYP(K_INDUCER_CHAIN, 4 * Mi * Cd * Cd, Mi * Cd * 6 + 4 * Cd * Cd, launch_gemm(g, s));
      }
      gecco_unpool_args u = {};
      u.q = w.big + 2 * C; u.ldq = C3; u.kv = khv_l; u.ldkv = 2 * C; u.v_off = C;
      u.clouds = clouds; u.rows_per_cloud = Np; u.heads = H; u.head_dim = hd; u.inducers = I;
      u.out_bf16 = w.y; u.ldo = C;
      u.vt_scratch = vt_l; u.vt_ready = kv_done ? 1 : 0;
      TRYP(K_UNPOOL_ATTN, 4 * Mv * I * Cd, Mv * Cd * 4 + Mi * Cd * 4, launch_unpool_attention(u, s));
      // x = x + out_proj(attn)  (:164), bf16 copy, statistics for mlp_norm
      g = gemm_base(w.y, C, L.out_w, C, rows, C, C, Np, points);
      g.bias = lw[GECCO_LW_UNPOOL_OUT_B];
      g.res = w.x; g.ldr = C; g.out_f32 = w.x; g.ldo32 = C;
      g.out_bf16 = xb_out; g.ldo16 = C;
      g.stats = stat(l, 3); g.stat_gs = C / sg;
      TRYP(K_GEMM_UNPOOL_OUT, 2 * Mv * Cd * Cd, Mv * Cd * 12 + 2 * Cd * Cd, launch_gemm(g, s));
    }
    // x = x + mlp(AdaGN_mlp(x, t))  (:165-166): mlp_norm folded into mlp.0; statistics for the next broadcast_norm /
    // the head norm
    double* const next_stats = (l + 1 < d.n_layers) ? stat(l + 1, 0) : head_stats;
    gecco_mlp_args mp = {};
    if (an) {
      mp.a = w.xb; mp.lda = C;
      mp.w1 = L.mlp_w0; mp.ldw1 = C; mp.b1 = lw[GECCO_LW_MLP_B0];
      mp.act_alpha = L.mlp_alpha; mp.act = act;
      mp.w2 = L.mlp_w2; mp.ldw2 = hid; mp.b2 = lw[GECCO_LW_MLP_B2];
      mp.m = rows; mp.c = C; mp.hidden = hid; mp.rows_per_cloud = Np; mp.valid_rows = points;
      mp.res = w.x; mp.ldr = C; mp.out_f32 = w.x; mp.ldo32 = C; mp.out_bf16 = xb_out; mp.ldo16 = C;
      mp.stats = next_stats; mp.stat_gs = C / sg;
      mp.anorm.stats = stat(l, 3); mp.anorm.stat_gs = C / sg; mp.anorm.groups = sg; mp.anorm.eps = 1e-5f;
      mp.anorm.t = w.c_noise; mp.anorm.t_stride = 1;
      mp.anorm.scale_w = lw[GECCO_LW_MN]; mp.anorm.scale_b = lw[GECCO_LW_MN + 1];
      mp.anorm.bias_w = lw[GECCO_LW_MN + 2]; mp.anorm.bias_b = lw[GECCO_LW_MN + 3];
      mp.scratch = w.big;  // k | v | q of this layer have been consumed
    }
    if (an && g_mlp_pair && mlp_pair_supported(mp)) {
      // one kernel: AdaGN on the A operand, the hidden tile of a row block parked in L2 between the products (mlp_pair.cu)
      TRYP(K_MLP_FUSED, 4 * Mv * Cd * Hd, Mv * Cd * 12 + 4 * Cd * Hd, launch_mlp_pair(mp, s));
    } else if (an) {
      gecco_gemm_args g = gemm_base(w.xb, C, L.mlp_w0, C, rows, hid, C, Np, points);
      set_anorm(g, lw + GECCO_LW_MN, stat(l, 3));
      g.bias = lw[GECCO_LW_MLP_B0]; g.bias_stride = 0; g.act = act; g.act_alpha = L.mlp_alpha;
      g.out_bf16 = w.big; g.ldo16 = hid;
      TRYP(K_GEMM_MLP0, 2 * Mv * Cd * Hd, Mv * (Cd * 2 + Hd * 2) + 2.0 * Cd * Hd, launch_gemm(g, s));
      g = gemm_base(w.big, hid, L.mlp_w2, hid, rows, C, hid, Np, points);
      g.bias = lw[GECCO_LW_MLP_B2];
      g.res = w.x; g.ldr = C; g.out_f32 = w.x; g.ldo32 = C;
      g.out_bf16 = xb_out; g.ldo16 = C;
      g.stats = next_stats; g.stat_gs = C / sg;
      TRYP(K_GEMM_MLP2, 2 * Mv * Cd * Hd, Mv * (Hd * 2 + Cd * 10) + 2 * Cd * Hd, launch_gemm(g, s));
    } else {
      gecco_fold_adagn_args f = fold_base(e, lw + GECCO_LW_MN, stat(l, 3), w.c_noise, clouds, points);
      f.w = lw[GECCO_LW_MLP_W0]; f.ldw = C; f.bias = lw[GECCO_LW_MLP_B0]; f.n_out = hid;
      f.w_folded_bf16 = w.wfold; f.ldwf = C; f.wf_cloud_stride = (long long)hid * C;
      f.bias_folded = w.bfold; f.bias_stride = hid;
      TRYP(K_FOLD_ADAGN, 2.0 * clouds * Hd * Cd, Hd * Cd * (4.0 + 2.0 * clouds), launch_fold_adagn(f, s));
      gecco_gemm_args g = gemm_base(w.xb, C, w.wfold, C, rows, hid, C, Np, points);
      g.w_rows_per_cloud = hid;
      g.bias = w.bfold; g.bias_stride = hid; g.act = act; g.act_alpha = L.mlp_alpha;
      g.out_bf16 = w.big; g.ldo16 = hid;
      TRYP(K_GEMM_MLP0, 2 * Mv * Cd * Hd, Mv * (Cd + Hd) * 2 + 2.0 * clouds * Cd * Hd, launch_gemm(g, s));
      g = gemm_base(w.big, hid, L.mlp_w2, hid, rows, C, hid, Np, points);
      g.bias = lw[GECCO_LW_MLP_B2];
      g.res = w.x; g.ldr = C; g.out_f32 = w.x; g.ldo32 = C;
      g.out_bf16 = w.xb; g.ldo16 = C;
      g.stats = next_stats; g.stat_gs = C / sg;
      TRYP(K_GEMM_MLP2, 2 * Mv * Cd * Hd, Mv * (Hd * 2 + Cd * 10) + 2 * Cd * Hd, launch_gemm(g, s));
    }
  }

  // ---------------------------------------------------------------- output head + EDM preconditioning / sampler update
  head.x = w.x; head.ldx = C;
  head.clouds = clouds; head.rows_per_cloud = Np; head.valid_rows = points; head.c = C;
  head.norm = d.head_norm; head.groups = d.head_groups; head.stats = head_stats; head.stat_gs = C / sg; head.eps = 1e-5f;
  head.w_out = e->net[GECCO_NW_OUT_W]; head.b_out = e->net[GECCO_NW_OUT_B];
  head.xin = xin;
  head.sigma = w.sigma_eff; head.sigma_stride = 1; head.sigma_data = sigma_data;
  TRYP(K_HEAD, 6 * Mv * Cd, Mv * (Cd * 4 + 60), launch_head(head, s));
  return GECCO_OK;
}

int check_common(const gecco_engine* e, int clouds, int points, const gecco_context& ctx, const void* ws, long long ws_bytes) {
  GECCO_REQUIRE(e != nullptr, "null engine handle");
  GECCO_REQUIRE(clouds > 0 && points > 0, "empty batch: clouds=%d points=%d", clouds, points);
  GECCO_REQUIRE(ws != nullptr && (reinterpret_cast<uintptr_t>(ws) & 255) == 0, "workspace must be a 256-byte aligned device buffer");
  const long long need = gecco_workspace_bytes(e, clouds, points);
  GECCO_REQUIRE(ws_bytes >= need, "workspace too small: %lld bytes given, %lld needed", ws_bytes, need);
  if (e->d.kind == 1) {
    GECCO_REQUIRE(ctx.K != nullptr, "conditional model: camera matrices K are required");
    for (int l = 0; l < e->d.n_levels; ++l)
      GECCO_REQUIRE(ctx.level_ptr[l] != nullptr && ctx.level_h[l] > 0 && ctx.level_w[l] > 0,
                    "conditional model: feature pyramid level %d is missing", l);
  }
  return GECCO_OK;
}

}  // namespace
}  // namespace gecco

using namespace gecco;

extern "C" int gecco_create(const gecco_model_desc* desc, const float* const* net_weights, const float* const* layer_weights,
                            void* stream, gecco_engine** out) {
  GECCO_REQUIRE(desc && net_weights && layer_weights && out, "gecco_create: null argument");
  const gecco_model_desc& d = *desc;
  const int C = d.feature_dim, H = d.num_heads, I = d.num_inducers, hid = d.mlp_hidden;
  GECCO_REQUIRE(d.kind == 0 || d.kind == 1, "gecco_create: unknown network kind %d", d.kind);
  GECCO_REQUIRE(d.n_layers >= 1 && d.n_layers <= GECCO_MAX_LAYERS, "gecco_create: n_layers out of range");
  GECCO_REQUIRE(C > 0 && C % 128 == 0 && C <= 1024, "gecco_create: feature_dim must be a multiple of 128 (<= 1024), got %d", C);
  GECCO_REQUIRE(H > 0 && C % H == 0 && (C / H == 32 || C / H == 48 || C / H == 64),
                "gecco_create: head dim must be 32, 48 or 64 (feature_dim %d, heads %d)", C, H);
  // whole blocks of 64 inducers (the query rows of one pool CTA, the key chunk of the unpool core), up to 256
  GECCO_REQUIRE(I >= 64 && I <= 256 && I % 64 == 0, "gecco_create: num_inducers must be 64, 128, 192 or 256 (got %d inducers)", I);
  // The GEMM epilogues keep the AdaGN statistics per group of C / adagn_groups channels; they are instantiated for the
  // widths that divide their 192-column panel.
  GECCO_REQUIRE(d.adagn_groups > 0 && C % d.adagn_groups == 0 && epi_stat_width_supported(C / d.adagn_groups),
                "gecco_create: feature_dim %d is not supported with %d AdaGN groups: the groups must be 4, 8, 12, 16, 24 or "
                "32 channels wide (feature_dim 128, 256, 384, 512, 768 or 1024 with 32 groups)", C, d.adagn_groups);
  GECCO_REQUIRE(hid > 0 && hid % 8 == 0, "gecco_create: mlp_hidden must be a multiple of 8");
  const int act = mlp_act_of(d.mlp_act);
  GECCO_REQUIRE(act == GECCO_ACT_GAUSSIAN || act == GECCO_ACT_GAUSSIAN_RAW || act == GECCO_ACT_RELU,
                "gecco_create: unknown MLP activation %d (supported: 1 normalised Gaussian, 2 raw Gaussian, 3 ReLU)", d.mlp_act);
  GECCO_REQUIRE(d.head_norm >= 0 && d.head_norm <= 2, "gecco_create: bad head_norm");
  GECCO_REQUIRE(d.head_norm != 2 || (d.head_groups > 0 && C % d.head_groups == 0 && (C / d.head_groups) % (C / d.adagn_groups) == 0),
                "gecco_create: head GroupNorm groups must be multiples of the AdaGN group width (%d channels)", C / d.adagn_groups);
  int ctot = 0;
  if (d.kind == 1) {
    GECCO_REQUIRE(d.n_levels >= 1 && d.n_levels <= GECCO_MAX_LEVELS, "gecco_create: 1..%d pyramid levels", GECCO_MAX_LEVELS);
    for (int l = 0; l < d.n_levels; ++l) {
      GECCO_REQUIRE(d.level_c[l] > 0 && d.level_c[l] % 8 == 0, "gecco_create: level channel counts must be multiples of 8");
      ctot += d.level_c[l];
    }
    GECCO_REQUIRE(d.img_groups > 0 && ctot % d.img_groups == 0, "gecco_create: image GroupNorm groups must divide %d", ctot);
    GECCO_REQUIRE(net_weights[GECCO_NW_IMG_W] && net_weights[GECCO_NW_IMG_B], "gecco_create: image projection weights missing");
  }
  for (int i : {GECCO_NW_EMBED_W, GECCO_NW_EMBED_B, GECCO_NW_OUT_W, GECCO_NW_OUT_B})
    GECCO_REQUIRE(net_weights[i] != nullptr, "gecco_create: network weight %d missing", i);
  for (int i = 0; i < d.n_layers * GECCO_LW_COUNT; ++i)
    GECCO_REQUIRE(layer_weights[i] != nullptr ||
                      (!act_is_gaussian(act) && (i % GECCO_LW_COUNT == GECCO_LW_BMLP_ALPHA || i % GECCO_LW_COUNT == GECCO_LW_MLP_ALPHA)), "gecco_create: layer weight %d (layer %d, slot %d) missing", i,
                  i / GECCO_LW_COUNT, i % GECCO_LW_COUNT);

  int dev = 0;
  cudaError_t ce = cudaGetDevice(&dev);
  if (ce != cudaSuccess) return fail_cuda(ce, "cudaGetDevice");
  if (int rc = gecco_init(dev)) return rc;

  gecco_engine* e = new (std::nothrow) gecco_engine();
  GECCO_REQUIRE(e != nullptr, "gecco_create: out of host memory");
  e->d = d;
  e->device = dev;
  for (int i = 0; i < GECCO_NW_COUNT; ++i) e->net[i] = net_weights[i];
  e->lw.assign(layer_weights, layer_weights + (size_t)d.n_layers * GECCO_LW_COUNT);
  e->layers.resize(d.n_layers);

  // bf16: pool out_proj, inducer mlp (2), unpool k/v in-proj, unpool out_proj, mlp.2, inducer queries
  const size_t per_layer_bf16 = (size_t)C * C + 2 * (size_t)hid * C + (size_t)2 * C * C + (size_t)C * C + (size_t)hid * C +
                                (size_t)H * I * (C / H) + (size_t)3 * C * C + (size_t)hid * C;
  // fp32: [kv_proj ; q in-proj] weight and bias (sources of the AdaGN fold)
  const size_t per_layer_f32 = (size_t)3 * C * C + (size_t)3 * C;
  size_t bytes = 0;
  for (int l = 0; l < d.n_layers; ++l) bytes += align_up(per_layer_bf16 * 2 + 64 * 32) + align_up(per_layer_f32 * 4 + 64 * 16);
  bytes += align_up((size_t)C * 4) + 4096;
  ce = cudaMalloc(&e->arena, bytes);
  if (ce != cudaSuccess) {
    delete e;
    return fail_cuda(ce, "cudaMalloc(packed weights)");
  }
  e->arena_bytes = bytes;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  Carver c{static_cast<uint8_t*>(e->arena)};
  auto pack = [&](const float* src, size_t n, float scale) -> __nv_bfloat16* {
    __nv_bfloat16* dst = c.take<__nv_bfloat16>(n);
    pack_bf16_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, dst, (long long)n, scale);
    return dst;
  };
  // softmax scale and the exp -> exp2 change of base folded into the query side of both attentions
  const float qscale = (float)(1.4426950408889634 / sqrt((double)(C / H)));
  std::vector<float> alphas(2 * d.n_layers, 0.f);  // ReLU reads no alpha
  for (int l = 0; l < d.n_layers; ++l) {
    const float* const* lw = layer_weights + (size_t)l * GECCO_LW_COUNT;
    gecco_engine::Layer& L = e->layers[l];
    L.pool_out_w = pack(lw[GECCO_LW_POOL_OUT_W], (size_t)C * C, 1.f);
    L.bmlp_w0 = pack(lw[GECCO_LW_BMLP_W0], (size_t)hid * C, 1.f);
    L.bmlp_w2 = pack(lw[GECCO_LW_BMLP_W2], (size_t)C * hid, 1.f);
    L.kv_w = pack(lw[GECCO_LW_UNPOOL_IN_W] + (size_t)C * C, (size_t)2 * C * C, 1.f);      // in_proj_weight[C:3C]
    L.out_w = pack(lw[GECCO_LW_UNPOOL_OUT_W], (size_t)C * C, 1.f);
    L.mlp_w2 = pack(lw[GECCO_LW_MLP_W2], (size_t)C * hid, 1.f);
    L.q_ind = pack(lw[GECCO_LW_INDUCERS], (size_t)H * I * (C / H), qscale);
    // [kv_proj.weight (2C rows, no bias) ; qscale * in_proj_weight[0:C] (bias qscale * in_proj_bias[0:C])]
    L.wcat = c.take<float>((size_t)3 * C * C);
    L.bcat = c.take<float>((size_t)3 * C);
    scale_add_f32_kernel<<<ceil_div(2 * C * C, 256), 256, 0, s>>>(lw[GECCO_LW_POOL_KV_W], nullptr, L.wcat, 2 * C * C, 1.f);
    scale_add_f32_kernel<<<ceil_div(C * C, 256), 256, 0, s>>>(lw[GECCO_LW_UNPOOL_IN_W], nullptr, L.wcat + (size_t)2 * C * C, C * C, qscale);
    cudaMemsetAsync(L.bcat, 0, (size_t)2 * C * sizeof(float), s);
    scale_add_f32_kernel<<<ceil_div(C, 256), 256, 0, s>>>(lw[GECCO_LW_UNPOOL_IN_B], nullptr, L.bcat + 2 * C, C, qscale);
    L.wcat16 = pack(L.wcat, (size_t)3 * C * C, 1.f);  // stream-ordered after the two kernels that fill wcat
    L.mlp_w0 = pack(lw[GECCO_LW_MLP_W0], (size_t)hid * C, 1.f);
    if (act_is_gaussian(act)) {
      cudaMemcpyAsync(&alphas[2 * l], lw[GECCO_LW_BMLP_ALPHA], sizeof(float), cudaMemcpyDeviceToHost, s);
      cudaMemcpyAsync(&alphas[2 * l + 1], lw[GECCO_LW_MLP_ALPHA], sizeof(float), cudaMemcpyDeviceToHost, s);
    }
  }
  e->img_bias = nullptr;
  if (d.kind == 1) {
    e->img_bias = c.take<float>(C);
    scale_add_f32_kernel<<<ceil_div(C, 256), 256, 0, s>>>(net_weights[GECCO_NW_IMG_B], net_weights[GECCO_NW_EMBED_B],
                                                          e->img_bias, C, 1.f);
  }
  ce = cudaStreamSynchronize(s);
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess || c.off > bytes) {
    cudaFree(e->arena);
    delete e;
    if (ce != cudaSuccess) return fail_cuda(ce, "gecco_create: weight packing");
    set_error("gecco_create: internal arena overflow");
    return GECCO_ERR_INVALID;
  }
  for (int l = 0; l < d.n_layers; ++l) {
    e->layers[l].bmlp_alpha = alphas[2 * l];
    e->layers[l].mlp_alpha = alphas[2 * l + 1];
  }
  *out = e;
  return GECCO_OK;
}

extern "C" int gecco_destroy(gecco_engine* e) {
  if (e == nullptr) return GECCO_OK;
  if (e->gstream != nullptr) cudaStreamSynchronize(e->gstream);
  for (auto& g : e->graphs) cudaGraphExecDestroy(g.exec);
  if (e->ev_fork != nullptr) cudaEventDestroy(e->ev_fork);
  if (e->ev_join != nullptr) cudaEventDestroy(e->ev_join);
  if (e->gstream != nullptr) cudaStreamDestroy(e->gstream);
  cudaFree(e->arena);
  delete e;
  return GECCO_OK;
}

extern "C" int64_t gecco_workspace_bytes(const gecco_engine* e, int32_t clouds, int32_t points) {
  if (e == nullptr || clouds <= 0 || points <= 0) return 0;
  return (int64_t)carve(e, clouds, points, nullptr).bytes;
}

extern "C" int gecco_denoise(gecco_engine* e, const gecco_denoise_args* a, void* stream) {
  GECCO_REQUIRE(a != nullptr, "gecco_denoise: null args");
  TRY(check_common(e, a->clouds, a->points, a->ctx, a->workspace, a->workspace_bytes));
  GECCO_REQUIRE(a->x != nullptr, "gecco_denoise: x is null");
  GECCO_REQUIRE(a->mode >= 0 && a->mode <= 3, "gecco_denoise: bad mode %d", a->mode);
  GECCO_REQUIRE(a->t_embed != nullptr || a->sigma != nullptr || a->sigma_imm > 0.f, "gecco_denoise: sigma missing");
  GECCO_REQUIRE(a->t_embed == nullptr || a->mode == 0, "gecco_denoise: a network-level call (t_embed) only supports mode 0");
  const Workspace w = carve(e, a->clouds, a->points, a->workspace);
  gecco_head_args h = {};
  h.mode = a->mode;
  h.out_f32 = a->out;
  h.x_hat = a->x_hat; h.x_next = a->x_next; h.d_cur = a->d_cur; h.xin_next = a->xin_next; h.noise_next = a->noise_next;
  h.t_hat = a->t_hat; h.t_next = a->t_next; h.churn_next = a->churn_next;
  return run_eval(e, w, a->x, a->sigma, a->sigma_stride, a->sigma_imm, a->t_embed, a->t_stride, a->clouds, a->points, a->ctx, a->cache_in,
                  a->cache_out, h, static_cast<cudaStream_t>(stream));
}

namespace gecco {
namespace {

int g_graphs_enabled = -1;  // -1: from the environment (GECCO_GRAPHS, default on)
bool graphs_enabled() {
  if (g_graphs_enabled < 0) {
    const char* v = getenv("GECCO_GRAPHS");
    g_graphs_enabled = (v != nullptr && v[0] == '0') ? 0 : 1;
  }
  return g_graphs_enabled != 0;
}

// Enqueues the whole sampler loop on `s` (also under stream capture: no host synchronisation, no allocation).
int enqueue_sample(gecco_engine* e, const gecco_sample_args* a, cudaStream_t s) {
  const Workspace w = carve(e, a->clouds, a->points, a->workspace);
  const long long n3 = (long long)a->clouds * a->points * 3;
  const double* t = a->host_t_steps;
  auto churn = [&](int i) {  // sqrt(t_hat^2 - t_cur^2) * S_noise  (diffusion.py:323-325)
    const double t_hat = t[i] + a->host_gamma[i] * t[i];
    return sqrt(t_hat * t_hat - t[i] * t[i]) * a->s_noise;
  };
  // x_hat_0 = latents * t_0 + churn_0 * noise_0  (:308, :325)
  // (a zero churn factor skips the noise read altogether: the deterministic sampler never touches the noise buffer)
  TRY(launch_sampler_init(a->latents, churn(0) != 0.0 ? a->noise : nullptr, t[0], churn(0), n3, w.x_hat, w.xin_a, s));
  for (int i = 0; i < a->num_steps; ++i) {
    const double t_hat = t[i] + a->host_gamma[i] * t[i];
    const double t_next = t[i + 1];
    gecco_head_args h = {};
    h.mode = 2;  // Euler (:335-336)
    h.x_hat = w.x_hat; h.x_next = w.x_next; h.d_cur = w.d_cur; h.xin_next = w.xin_b;
    h.t_hat = t_hat; h.t_next = t_next;
    TRY(run_eval(e, w, w.xin_a, nullptr, 0, (float)t_hat, nullptr, 0, a->clouds, a->points, a->ctx, nullptr, nullptr, h, s));
    if (i < a->num_steps - 1) {  // Heun (:339-347) + churn of step i+1
      h.mode = 3;
      h.xin_next = w.xin_a;
      h.churn_next = churn(i + 1);
      h.noise_next = h.churn_next != 0.0 ? a->noise + (size_t)(i + 1) * n3 : nullptr;
      TRY(run_eval(e, w, w.xin_b, nullptr, 0, (float)t_next, nullptr, 0, a->clouds, a->points, a->ctx, nullptr, nullptr, h, s));
    }
  }
  // the last step is Euler only: the result is x_next
  copy_f64_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, s>>>(w.x_next, a->x_out, n3);
  GECCO_CHECK_LAUNCH("copy_f64_kernel");
  return GECCO_OK;
}

// Everything a captured sampler graph depends on: shapes, schedule (baked into kernel arguments) and every pointer.
std::vector<unsigned char> sample_key(const gecco_sample_args* a) {
  std::vector<unsigned char> k;
  auto put = [&](const void* p, size_t n) { k.insert(k.end(), (const unsigned char*)p, (const unsigned char*)p + n); };
  put(&a->clouds, sizeof(int32_t)); put(&a->points, sizeof(int32_t)); put(&a->num_steps, sizeof(int32_t));
  put(a->host_t_steps, sizeof(double) * (a->num_steps + 1));
  put(a->host_gamma, sizeof(double) * a->num_steps);
  put(&a->s_noise, sizeof(double));
  put(&a->latents, sizeof(void*)); put(&a->noise, sizeof(void*)); put(&a->x_out, sizeof(void*));
  put(&a->ctx, sizeof(gecco_context));
  put(&a->workspace, sizeof(void*)); put(&a->workspace_bytes, sizeof(int64_t));
  const int options = g_anorm | (g_chain << 1) | (g_mlp_pair << 2);
  put(&options, sizeof(int));
  return k;
}

// sampler loops (one graph per argument set) and upsampling steps (one graph per noise level: 64 per schedule)
constexpr size_t kMaxGraphs = 160;

void drop_graph(gecco_engine* e, size_t i) {
  cudaGraphExecDestroy(e->graphs[i].exec);
  e->graphs.erase(e->graphs.begin() + i);
}

}  // namespace
void set_graphs_option(int value) { g_graphs_enabled = value != 0 ? 1 : 0; }
void set_anorm_option(int value) { g_anorm = value != 0 ? 1 : 0; }
void set_chain_option(int value) { g_chain = value != 0 ? 1 : 0; }
void set_mlp_pair_option(int value) { g_mlp_pair = value != 0 ? 1 : 0; }
}  // namespace gecco

namespace gecco {
namespace {
// Runs `enqueue(stream)` through the engine's CUDA-graph cache: captured on the engine's own stream the first time `key`
// is seen (forked from / joined to the caller's stream with events, so the legacy default stream works too), replayed
// afterwards.  Falls back to a plain enqueue when graphs are off, while profiling, or when the caller's stream is itself
// being captured.
template <typename Enqueue>
int run_graphed(gecco_engine* e, const std::vector<unsigned char>& key, cudaStream_t s, Enqueue enqueue) {
  e->last_graph_status = 0;
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (s != nullptr && s != cudaStreamLegacy) cudaStreamIsCapturing(s, &cap);
  if (!graphs_enabled() || g_prof.on || cap != cudaStreamCaptureStatusNone) return enqueue(s);
  if (e->gstream == nullptr) {
    cudaError_t ce = cudaStreamCreateWithFlags(&e->gstream, cudaStreamNonBlocking);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming);
    if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&e->ev_join, cudaEventDisableTiming);
    if (ce != cudaSuccess) return fail_cuda(ce, "graph stream / events");
  }
  size_t hit = e->graphs.size();
  for (size_t i = 0; i < e->graphs.size(); ++i)
    if (e->graphs[i].key == key) { hit = i; break; }
  if (hit == e->graphs.size()) {
    // capture (thread-local mode: other threads' CUDA calls neither join nor invalidate it)
    const long long before = g_launches;
    cudaError_t ce = cudaStreamBeginCapture(e->gstream, cudaStreamCaptureModeThreadLocal);
    if (ce != cudaSuccess) return fail_cuda(ce, "cudaStreamBeginCapture");
    const int rc = enqueue(e->gstream);
    cudaGraph_t graph = nullptr;
    ce = cudaStreamEndCapture(e->gstream, &graph);
    const long long launches = g_launches - before;
    g_launches = before;  // counted per replay below
    cudaGraphExec_t exec = nullptr;
    if (rc == GECCO_OK && ce == cudaSuccess && graph != nullptr) ce = cudaGraphInstantiate(&exec, graph, 0);
    if (graph != nullptr) cudaGraphDestroy(graph);
    if (rc != GECCO_OK) return rc;  // argument errors surface exactly as in the eager path
    if (ce != cudaSuccess || exec == nullptr) {
      // a driver that cannot capture this launch sequence: run eagerly, visibly (gecco_graph_status < 0)
      cudaGetLastError();
      const int rc2 = enqueue(s);
      e->last_graph_status = -1;
      return rc2;
    }
    if (e->graphs.size() >= kMaxGraphs) {
      size_t oldest = 0;
      for (size_t i = 1; i < e->graphs.size(); ++i)
        if (e->graphs[i].stamp < e->graphs[oldest].stamp) oldest = i;
      drop_graph(e, oldest);
    }
    e->graphs.push_back({key, exec, launches, 0});
    hit = e->graphs.size() - 1;
    e->last_graph_status = 1;
  } else {
    e->last_graph_status = 2;
  }
  gecco_engine::SampleGraph& g = e->graphs[hit];
  g.stamp = ++e->graph_clock;
  cudaError_t ce = cudaEventRecord(e->ev_fork, s);
  if (ce == cudaSuccess) ce = cudaStreamWaitEvent(e->gstream, e->ev_fork, 0);
  if (ce == cudaSuccess) ce = cudaGraphLaunch(g.exec, e->gstream);
  if (ce == cudaSuccess) ce = cudaEventRecord(e->ev_join, e->gstream);
  if (ce == cudaSuccess) ce = cudaStreamWaitEvent(s, e->ev_join, 0);
  if (ce != cudaSuccess) return fail_cuda(ce, "graph launch");
  g_launches += g.launches;
  return GECCO_OK;
}
}  // namespace
}  // namespace gecco

extern "C" int gecco_sample(gecco_engine* e, const gecco_sample_args* a, void* stream) {
  GECCO_REQUIRE(a != nullptr, "gecco_sample: null args");
  TRY(check_common(e, a->clouds, a->points, a->ctx, a->workspace, a->workspace_bytes));
  GECCO_REQUIRE(a->num_steps >= 1 && a->host_t_steps && a->host_gamma, "gecco_sample: schedule missing");
  GECCO_REQUIRE(a->latents && a->x_out, "gecco_sample: latents / output missing");
  for (int i = 0; i < a->num_steps; ++i)
    GECCO_REQUIRE(a->noise != nullptr || a->host_gamma[i] == 0.0 || a->s_noise == 0.0, "gecco_sample: noise missing (gamma[%d] > 0)", i);
  return run_graphed(e, sample_key(a), static_cast<cudaStream_t>(stream), [&](cudaStream_t s) { return enqueue_sample(e, a, s); });
}

// ------------------------------------------------------------------------------------------------ upsampling
namespace gecco {
namespace {
struct UpsampleLayout {
  size_t carve_bytes, cache_off, seed_in_off, seed_out_off, khv_off, vt_off, total;
};
UpsampleLayout upsample_layout(const gecco_engine* e, int clouds, int seed_points, int new_points) {
  UpsampleLayout u;
  const int big = seed_points > new_points ? seed_points : new_points;
  u.carve_bytes = carve(e, clouds, big, nullptr).bytes;
  size_t off = align_up(u.carve_bytes);
  u.cache_off = off;
  off = align_up(off + (size_t)e->d.n_layers * clouds * e->d.num_inducers * e->d.feature_dim * sizeof(float));
  u.seed_in_off = off;
  off = align_up(off + (size_t)clouds * seed_points * 3 * sizeof(float));
  u.seed_out_off = off;
  off = align_up(off + (size_t)clouds * seed_points * 3 * sizeof(float));
  u.khv_off = off;
  off = align_up(off + (size_t)e->d.n_layers * clouds * e->d.num_inducers * 2 * e->d.feature_dim * sizeof(__nv_bfloat16));
  u.vt_off = off;
  off = align_up(off + (size_t)e->d.n_layers * clouds * e->d.num_inducers * e->d.feature_dim * sizeof(__nv_bfloat16));
  u.total = off;
  return u;
}
}  // namespace
}  // namespace gecco

extern "C" int64_t gecco_upsample_workspace_bytes(const gecco_engine* e, int32_t clouds, int32_t seed_points, int32_t new_points) {
  if (e == nullptr || clouds <= 0 || seed_points <= 0 || new_points <= 0) return 0;
  return (int64_t)upsample_layout(e, clouds, seed_points, new_points).total;
}

namespace gecco {
namespace {
int enqueue_upsample_step(gecco_engine* e, const gecco_upsample_step_args* a, cudaStream_t s);
}
}  // namespace gecco

extern "C" int gecco_upsample_step(gecco_engine* e, const gecco_upsample_step_args* a, void* stream) {
  GECCO_REQUIRE(a != nullptr, "gecco_upsample_step: null args");
  GECCO_REQUIRE(e != nullptr, "null engine handle");
  GECCO_REQUIRE(a->seed_points > 0 && a->new_points > 0 && a->num_substeps >= 1, "gecco_upsample_step: empty problem");
  GECCO_REQUIRE(a->seed_data && a->seed_noise && a->noise && a->x, "gecco_upsample_step: seed / noise / state missing");
  GECCO_REQUIRE(a->t_cur > 0.0, "gecco_upsample_step: t_cur must be positive");
  const UpsampleLayout u = upsample_layout(e, a->clouds, a->seed_points, a->new_points);
  TRY(check_common(e, a->clouds, a->new_points, a->ctx, a->workspace, a->workspace_bytes));
  GECCO_REQUIRE(a->workspace_bytes >= (int64_t)u.total, "workspace too small: %lld bytes given, %lld needed",
                (long long)a->workspace_bytes, (long long)u.total);
  // everything the launch sequence depends on (the struct holds shapes, schedule scalars and every pointer)
  std::vector<unsigned char> key(sizeof(gecco_upsample_step_args) + 8);
  memcpy(key.data(), a, sizeof(gecco_upsample_step_args));
  memcpy(key.data() + sizeof(gecco_upsample_step_args), "upsample", 8);
  key.push_back((unsigned char)(g_anorm | (g_chain << 1) | (g_mlp_pair << 2)));
  return run_graphed(e, key, static_cast<cudaStream_t>(stream), [&](cudaStream_t s) { return enqueue_upsample_step(e, a, s); });
}

namespace gecco {
namespace {
int enqueue_upsample_step(gecco_engine* e, const gecco_upsample_step_args* a, cudaStream_t s) {
  const UpsampleLayout u = upsample_layout(e, a->clouds, a->seed_points, a->new_points);
  uint8_t* base = static_cast<uint8_t*>(a->workspace);
  float* cache = reinterpret_cast<float*>(base + u.cache_off);
  float* seed_in = reinterpret_cast<float*>(base + u.seed_in_off);
  float* seed_out = reinterpret_cast<float*>(base + u.seed_out_off);
  KvCache kv_write = {reinterpret_cast<__nv_bfloat16*>(base + u.khv_off), reinterpret_cast<__nv_bfloat16*>(base + u.vt_off), 1};
  KvCache kv_read = kv_write;
  kv_read.mode = 2;
  const long long ns = (long long)a->clouds * a->seed_points * 3, n3 = (long long)a->clouds * a->new_points * 3;
  // data_ctx = data + randn * t_cur; full evaluation on the seed cloud, inducer states cached (:430-437)
  TRY(launch_seed_renoise(a->seed_data, a->seed_noise, (float)a->t_cur, ns, seed_in, s));
  {
    const Workspace ws = carve(e, a->clouds, a->seed_points, a->workspace);
    gecco_head_args h = {};
    h.mode = 1;
    h.out_f32 = seed_out;  // the denoised seed cloud itself is not used (:431 `_`)
    TRY(run_eval(e, ws, seed_in, nullptr, 0, (float)a->t_cur, nullptr, 0, a->clouds, a->seed_points, a->ctx, nullptr, cache, h, s, &kv_write));
  }
  const Workspace w = carve(e, a->clouds, a->new_points, a->workspace);
  const double t_hat = a->t_cur + a->gamma * a->t_cur;
  const float churn = (float)(sqrt(t_hat * t_hat - a->t_cur * a->t_cur) * a->s_noise);
  const float redo = a->last_step ? 0.f : (float)sqrt(a->t_cur * a->t_cur - a->t_next * a->t_next);
  const double* src = a->x;
  for (int uu = 0; uu < a->num_substeps; ++uu) {
    const float* n_churn = a->noise + (size_t)(a->last_step ? uu : 2 * uu) * n3;
    const float* n_redo = (uu > 0 && !a->last_step) ? a->noise + (size_t)(2 * uu - 1) * n3 : nullptr;  // of the previous sub-step
    TRY(launch_substep_noise(src, n_redo, redo, n_churn, churn, n3, w.x_hat, w.xin_a, s));
    gecco_head_args h = {};
    h.mode = 2;  // Euler (:452-454)
    h.x_hat = w.x_hat; h.x_next = w.x_next; h.d_cur = w.d_cur; h.xin_next = w.xin_b;
    h.t_hat = t_hat; h.t_next = a->t_next;
    TRY(run_eval(e, w, w.xin_a, nullptr, 0, (float)t_hat, nullptr, 0, a->clouds, a->new_points, a->ctx, cache, nullptr, h, s, kv_read.mode == 2 ? &kv_read : nullptr));
    if (!a->last_step) {  // 2nd order correction (:457-460); the result replaces x_hat
      h.mode = 3;
      h.xin_next = w.xin_a;
      h.noise_next = nullptr; h.churn_next = 0.0;
      TRY(run_eval(e, w, w.xin_b, nullptr, 0, (float)a->t_next, nullptr, 0, a->clouds, a->new_points, a->ctx, cache, nullptr, h, s, kv_read.mode == 2 ? &kv_read : nullptr));
      src = w.x_hat;
    } else {
      src = w.x_next;
    }
  }
  copy_f64_kernel<<<(unsigned)((n3 + 255) / 256), 256, 0, s>>>(src, a->x, n3);
  GECCO_CHECK_LAUNCH("copy_f64_kernel");
  return GECCO_OK;
}
}  // namespace
}  // namespace gecco

extern "C" int gecco_graph_status(const gecco_engine* e) { return e ? e->last_graph_status : 0; }

// ------------------------------------------------------------------------------------------------ profiling
extern "C" int gecco_profile_start(void) {
  g_prof.on = true;
  g_prof.used = 0;
  g_prof.recs.clear();
  return GECCO_OK;
}

extern "C" int gecco_profile_stop(gecco_profile_entry* out, int32_t capacity, int32_t* count) {
  g_prof.on = false;
  cudaError_t ce = cudaDeviceSynchronize();
  if (ce != cudaSuccess) return fail_cuda(ce, "gecco_profile_stop: cudaDeviceSynchronize");
  gecco_profile_entry acc[K_COUNT];
  memset(acc, 0, sizeof(acc));
  for (int i = 0; i < K_COUNT; ++i) strncpy(acc[i].name, kClassNames[i], sizeof(acc[i].name) - 1);
  for (const Profiler::Rec& r : g_prof.recs) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, g_prof.pool[r.ev], g_prof.pool[r.ev + 1]) != cudaSuccess) continue;
    acc[r.cls].launches += 1;
    acc[r.cls].ms += ms;
    acc[r.cls].flops += r.flops;
    acc[r.cls].bytes += r.bytes;
  }
  g_prof.recs.clear();
  g_prof.used = 0;
  int n = 0;
  for (int i = 0; i < K_COUNT; ++i) {
    if (acc[i].launches == 0) continue;
    if (out != nullptr && n < capacity) out[n] = acc[i];
    ++n;
  }
  if (count != nullptr) *count = n;
  return GECCO_OK;
}
