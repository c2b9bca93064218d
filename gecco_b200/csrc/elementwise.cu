// HBM-bound row-wise kernels around the tensor-core GEMMs:
//   group statistics, AdaGN apply (fp32 -> bf16 operand), unconditional lift, output head + EDM step,
//   reparametrisations.  All are coalesced over the channel dimension (one float4 per thread).
#include "common.cuh"
#include "ptx.cuh"
#include "norm.cuh"

#include <stdlib.h>

namespace gecco {

namespace {

// ------------------------------------------------------------------------------------------------
// Group statistics: stats[cloud][c / gs][{sum, sumsq}] over the valid rows of each cloud (double).
// grid (row chunks, clouds), block C/4 threads (looping if C/4 > blockDim).
constexpr int STAT_ROWS = 64;

__global__ void group_stats_kernel(const float* __restrict__ x, long long ldx, int rows_per_cloud, int valid_rows,
                                   int C, int gs, double* __restrict__ stats) {
  // [C/gs][2] per-block partial sums.  Double: the shared-memory atomics arrive in any order, and fp32 partials would
  // make the statistics (and everything folded from them) differ in the last bit from run to run.
  extern __shared__ double sgrp_d[];
  double* sgrp = sgrp_d;
  const int ngroups = C / gs;
  for (int i = threadIdx.x; i < ngroups * 2; i += blockDim.x) sgrp[i] = 0.0;
  __syncthreads();
  const int cloud = blockIdx.y;
  const int r0 = blockIdx.x * STAT_ROWS;
  const int r1 = min(r0 + STAT_ROWS, valid_rows);
  const float* base = x + ((long long)cloud * rows_per_cloud) * ldx;
  for (int cq = threadIdx.x; cq < C / 4; cq += blockDim.x) {
    float s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    for (int r = r0; r < r1; ++r) {
      const float4 v = *reinterpret_cast<const float4*>(base + (long long)r * ldx + cq * 4);
      s1[0] += v.x; s2[0] += v.x * v.x;
      s1[1] += v.y; s2[1] += v.y * v.y;
      s1[2] += v.z; s2[2] += v.z * v.z;
      s1[3] += v.w; s2[3] += v.w * v.w;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int g = (cq * 4 + j) / gs;
      atomicAdd(&sgrp[g * 2], static_cast<double>(s1[j]));
      atomicAdd(&sgrp[g * 2 + 1], static_cast<double>(s2[j]));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < ngroups * 2; i += blockDim.x)
    atomicAdd(stats + (long long)cloud * ngroups * 2 + i, sgrp[i]);
}

// ------------------------------------------------------------------------------------------------
// AdaGN apply (models/normalization.py:36-44): y = scale(t) * (x - mean_g) * rstd_g + bias(t)
// with scale(t) = t . scale_w[c, :] + scale_b[c] (same for bias).  Padding rows are written as 0.
constexpr int ADAGN_ROWS = 8;  // rows per block: the inducer side has only 64 rows per cloud, small blocks fill the SMs

__global__ void adagn_apply_kernel(const float* __restrict__ x, long long ldx, const double* __restrict__ stats,
                                   int stat_gs, const float* __restrict__ t, int t_stride, int ctx_dim,
                                   const float* __restrict__ scale_w, const float* __restrict__ scale_b,
                                   const float* __restrict__ bias_w, const float* __restrict__ bias_b,
                                   int rows_per_cloud, int valid_rows, int C, int groups, float eps,
                                   __nv_bfloat16* __restrict__ out16, long long ldo16, float* __restrict__ out32,
                                   long long ldo32) {
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  const int cloud = blockIdx.y;
  const int r0 = blockIdx.x * ADAGN_ROWS;
  const int gs = C / groups;
  const double count = static_cast<double>(valid_rows) * gs;
  const double* cstats = stats + (long long)cloud * (C / stat_gs) * 2;
  const long long row_base = (long long)cloud * rows_per_cloud;
  for (int cq = threadIdx.x; cq < C / 4; cq += blockDim.x) {
    // the rows of this thread are loaded first: their latency overlaps the (double precision) statistics below
    float4 xv[ADAGN_ROWS];
#pragma unroll
    for (int i = 0; i < ADAGN_ROWS; ++i) {
      const int r = r0 + i;
      xv[i] = (r < valid_rows && r < rows_per_cloud)
                  ? __ldg(reinterpret_cast<const float4*>(x + (row_base + r) * ldx + cq * 4))
                  : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    float a[4], s[4];
    float mean = 0.f, rstd = 0.f;
    int g_prev = -1;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = cq * 4 + j;
      if (c / gs != g_prev) {  // once per thread when the group size is a multiple of 4
        g_prev = c / gs;
        group_mean_rstd(cstats, g_prev, gs, stat_gs, count, eps, mean, rstd);
      }
      float sc = __ldg(scale_b + c), bi = __ldg(bias_b + c);
      for (int i = 0; i < ctx_dim; ++i) {
        const float ti = __ldg(t + (long long)cloud * t_stride + i);
        sc += ti * __ldg(scale_w + (long long)c * ctx_dim + i);
        bi += ti * __ldg(bias_w + (long long)c * ctx_dim + i);
      }
      a[j] = sc * rstd;
      s[j] = bi - sc * rstd * mean;
    }
#pragma unroll
    for (int i = 0; i < ADAGN_ROWS; ++i) {
      const int r = r0 + i;
      if (r >= rows_per_cloud) break;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (r < valid_rows) {
        v.x = a[0] * xv[i].x + s[0];
        v.y = a[1] * xv[i].y + s[1];
        v.z = a[2] * xv[i].z + s[2];
        v.w = a[3] * xv[i].w + s[3];
      }
      if (out16 != nullptr) {
        uint2 pk = make_uint2(pack_bf16x2(v.x, v.y), pack_bf16x2(v.z, v.w));
        *reinterpret_cast<uint2*>(out16 + (row_base + r) * ldo16 + cq * 4) = pk;
      }
      if (out32 != nullptr) *reinterpret_cast<float4*>(out32 + (row_base + r) * ldo32 + cq * 4) = v;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// AdaGN followed by a Linear, folded per cloud (models/normalization.py:36-44 + the consumer nn.Linear):
//   AdaGN(x)[c] = a[c] x[c] + s[c],  a = scale(t) rstd_g,  s = bias(t) - a mean_g
//   Linear(AdaGN(x))[o] = sum_c (W[o,c] a[c]) x[c] + (b[o] + sum_c W[o,c] s[c])
// so the consumer GEMM reads the bf16 residual stream directly with per-cloud weights.  grid (row blocks, clouds),
// 256 threads; a warp owns whole output rows (coalesced fp32 reads, 8 B bf16 writes, shuffle-reduced bias dot).
constexpr int FOLD_ROWS = 48;    // output rows per block
constexpr int FOLD_CLOUDS = 4;   // clouds per block: every fp32 weight row is read once and folded for all of them
constexpr int FOLD_MAXC = 1024;
constexpr int FOLD_THREADS = 256;

__global__ void __launch_bounds__(FOLD_THREADS)
fold_adagn_kernel(const float* __restrict__ W, long long ldw, const float* __restrict__ bias, int n_out, int C,
                  const double* __restrict__ stats, int stat_gs, int groups, double count, float eps,
                  const float* __restrict__ t, int t_stride, const float* __restrict__ scale_w,
                  const float* __restrict__ scale_b, const float* __restrict__ bias_w, const float* __restrict__ bias_b,
                  int clouds, __nv_bfloat16* __restrict__ wf, long long ldwf, long long wf_cloud_stride,
                  float* __restrict__ bf, int bf_stride) {
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  extern __shared__ __align__(16) float fold_smem[];
  float* sa = fold_smem;                      // [FOLD_CLOUDS][C]
  float* ss = sa + FOLD_CLOUDS * C;           // [FOLD_CLOUDS][C]
  float* smean = ss + FOLD_CLOUDS * C;        // [FOLD_CLOUDS][groups]
  float* srstd = smean + FOLD_CLOUDS * groups;
  const int cloud0 = blockIdx.y * FOLD_CLOUDS;
  const int ncl = min(FOLD_CLOUDS, clouds - cloud0);
  const int gs = C / groups;
  // group statistics once per (cloud, group) (the only double precision arithmetic), then per-channel coefficients
  for (int i = threadIdx.x; i < ncl * groups; i += blockDim.x) {
    const int cl = i / groups, g = i - cl * groups;
    float mean, rstd;
    group_mean_rstd(stats + (long long)(cloud0 + cl) * (C / stat_gs) * 2, g, gs, stat_gs, count, eps, mean, rstd);
    smean[i] = mean;
    srstd[i] = rstd;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < ncl * C; i += blockDim.x) {
    const int cl = i / C, c = i - cl * C;
    const int g = c / gs;
    const float tc = __ldg(t + (long long)(cloud0 + cl) * t_stride);
    const float sc = tc * __ldg(scale_w + c) + __ldg(scale_b + c);
    const float bi = tc * __ldg(bias_w + c) + __ldg(bias_b + c);
    const float a = sc * srstd[cl * groups + g];
    sa[i] = a;
    ss[i] = bi - a * smean[cl * groups + g];
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int o_end = min((int)(blockIdx.x + 1) * FOLD_ROWS, n_out);
  constexpr int NW = FOLD_THREADS / 32;
  constexpr int ILP = 2;  // weight rows in flight per warp
  for (int ob = blockIdx.x * FOLD_ROWS + warp; ob < o_end; ob += NW * ILP) {
    float dot[ILP][FOLD_CLOUDS];
#pragma unroll
    for (int u = 0; u < ILP; ++u)
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) dot[u][cl] = 0.f;
    for (int c = lane * 4; c < C; c += 128) {
      float4 w[ILP];
#pragma unroll
      for (int u = 0; u < ILP; ++u) {
        const int o = ob + u * NW;
        w[u] = o < o_end ? __ldg(reinterpret_cast<const float4*>(W + (long long)o * ldw + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
      }
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) {
        if (cl >= ncl) break;
        const float4 a = *reinterpret_cast<const float4*>(sa + cl * C + c);
        const float4 sv = *reinterpret_cast<const float4*>(ss + cl * C + c);
#pragma unroll
        for (int u = 0; u < ILP; ++u) {
          const int o = ob + u * NW;
          if (o < o_end) {
            dot[u][cl] += w[u].x * sv.x + w[u].y * sv.y + w[u].z * sv.z + w[u].w * sv.w;
            *reinterpret_cast<uint2*>(wf + (long long)(cloud0 + cl) * wf_cloud_stride + (long long)o * ldwf + c) =
                make_uint2(pack_bf16x2(w[u].x * a.x, w[u].y * a.y), pack_bf16x2(w[u].z * a.z, w[u].w * a.w));
          }
        }
      }
    }
#pragma unroll
    for (int u = 0; u < ILP; ++u) {
      const int o = ob + u * NW;
      const float b0 = (bias != nullptr && o < o_end) ? __ldg(bias + o) : 0.f;
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) {
        const float d = warp_sum(dot[u][cl]);
        if (lane == 0 && o < o_end && cl < ncl) bf[(long long)(cloud0 + cl) * bf_stride + o] = d + b0;
      }
    }
  }
}

// Same fold, specialised for C = 128 NSTEP (384 on this path) with the weight rows held in registers: a warp owns
// FOLD_ROWS / 8 = 6 rows in two halves of 3; the 9 float4 loads of a half are issued together, the first half BEFORE the
// prologue (the weights do not depend on the statistics), so the L2 latency of the weights is paid twice per warp under
// other work instead of nine times in sequence as in the generic kernel (24 -> see DESIGN.md for the measured time).
template <int NSTEP>
__global__ void __launch_bounds__(FOLD_THREADS, 2)
fold_adagn_fast_kernel(const float* __restrict__ W, long long ldw, const float* __restrict__ bias, int n_out,
                       const double* __restrict__ stats, int stat_gs, int groups, double count, float eps,
                       const float* __restrict__ t, int t_stride, const float* __restrict__ scale_w,
                       const float* __restrict__ scale_b, const float* __restrict__ bias_w, const float* __restrict__ bias_b,
                       int clouds, __nv_bfloat16* __restrict__ wf, long long ldwf, long long wf_cloud_stride,
                       float* __restrict__ bf, int bf_stride) {
  constexpr int C = 128 * NSTEP;
  constexpr int NW = FOLD_THREADS / 32;
  constexpr int HALF = FOLD_ROWS / NW / 2;  // 3 rows per half
  extern __shared__ __align__(16) float fold_smem[];
  float* sa = fold_smem;                      // [FOLD_CLOUDS][C]
  float* ss = sa + FOLD_CLOUDS * C;           // [FOLD_CLOUDS][C]
  float* smean = ss + FOLD_CLOUDS * C;        // [FOLD_CLOUDS][groups]
  float* srstd = smean + FOLD_CLOUDS * groups;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cloud0 = blockIdx.y * FOLD_CLOUDS;
  const int ncl = min(FOLD_CLOUDS, clouds - cloud0);
  const int row0 = blockIdx.x * FOLD_ROWS + warp;  // rows row0 + NW i, i < 6
  auto load_half = [&](int h, float4 (&w)[HALF][NSTEP]) {
#pragma unroll
    for (int i = 0; i < HALF; ++i) {
      const int o = row0 + (h * HALF + i) * NW;
#pragma unroll
      for (int j = 0; j < NSTEP; ++j)
        w[i][j] = o < n_out ? __ldg(reinterpret_cast<const float4*>(W + (long long)o * ldw + lane * 4 + 128 * j))
                            : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  float4 w[HALF][NSTEP];
  load_half(0, w);  // weights are constants: in flight across the wait on the predecessor and the prologue
  pdl_wait();       // programmatic dependent launch: the predecessor (producer of the statistics) has completed
  pdl_launch_dependents();
  const int gs = C / groups;
  for (int i = threadIdx.x; i < ncl * groups; i += blockDim.x) {
    const int cl = i / groups, g = i - cl * groups;
    float mean, rstd;
    group_mean_rstd(stats + (long long)(cloud0 + cl) * (C / stat_gs) * 2, g, gs, stat_gs, count, eps, mean, rstd);
    smean[i] = mean;
    srstd[i] = rstd;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < ncl * C; i += blockDim.x) {
    const int cl = i / C, c = i - cl * C;
    const int g = c / gs;
    const float tc = __ldg(t + (long long)(cloud0 + cl) * t_stride);
    const float sc = tc * __ldg(scale_w + c) + __ldg(scale_b + c);
    const float bi = tc * __ldg(bias_w + c) + __ldg(bias_b + c);
    const float a = sc * srstd[cl * groups + g];
    sa[i] = a;
    ss[i] = bi - a * smean[cl * groups + g];
  }
  __syncthreads();
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    if (h == 1) load_half(1, w);
    float dot[HALF][FOLD_CLOUDS];
#pragma unroll
    for (int i = 0; i < HALF; ++i)
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) dot[i][cl] = 0.f;
#pragma unroll
    for (int j = 0; j < NSTEP; ++j) {
      const int c = lane * 4 + 128 * j;
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) {
        if (cl >= ncl) break;
        const float4 a = *reinterpret_cast<const float4*>(sa + cl * C + c);
        const float4 sv = *reinterpret_cast<const float4*>(ss + cl * C + c);
        __nv_bfloat16* dst = wf + (long long)(cloud0 + cl) * wf_cloud_stride + c;
#pragma unroll
        for (int i = 0; i < HALF; ++i) {
          const int o = row0 + (h * HALF + i) * NW;
          if (o < n_out) {
            const float4 wv = w[i][j];
            dot[i][cl] += wv.x * sv.x + wv.y * sv.y + wv.z * sv.z + wv.w * sv.w;
            *reinterpret_cast<uint2*>(dst + (long long)o * ldwf) =
                make_uint2(pack_bf16x2(wv.x * a.x, wv.y * a.y), pack_bf16x2(wv.z * a.z, wv.w * a.w));
          }
        }
      }
    }
#pragma unroll
    for (int i = 0; i < HALF; ++i) {
      const int o = row0 + (h * HALF + i) * NW;
      const float b0 = (bias != nullptr && o < n_out) ? __ldg(bias + o) : 0.f;
#pragma unroll
      for (int cl = 0; cl < FOLD_CLOUDS; ++cl) {
        const float d = warp_sum(dot[i][cl]);
        if (lane == 0 && o < n_out && cl < ncl) bf[(long long)(cloud0 + cl) * bf_stride + o] = d + b0;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Unconditional lift (models/linear_lift.py:21,44): x = W (c_in * xin) + b, plus AdaGN statistics of x
// at `gs`-channel granularity.  Padding rows are written as 0.
constexpr int LIFT_ROWS = 32;

__global__ void lift_kernel(const float* __restrict__ xin, const float* __restrict__ sigma, int sigma_stride,
                            float sigma_data, const float* __restrict__ w, const float* __restrict__ b,
                            int rows_per_cloud, int valid_rows, int C, int gs, float* __restrict__ x, long long ldx,
                            __nv_bfloat16* __restrict__ xb, long long ldxb, double* __restrict__ stats) {
  extern __shared__ double sgrp_d[];  // double partials: order-independent in practice (see group_stats_kernel)
  double* sgrp = sgrp_d;
  const int ngroups = C / gs;
  for (int i = threadIdx.x; i < ngroups * 2; i += blockDim.x) sgrp[i] = 0.0;
  __syncthreads();
  const int cloud = blockIdx.y;
  const int r0 = blockIdx.x * LIFT_ROWS;
  const int r1 = min(r0 + LIFT_ROWS, rows_per_cloud);
  float c_in = 1.f;
  if (sigma != nullptr) {
    const float sg = __ldg(sigma + (long long)cloud * sigma_stride);
    c_in = 1.0f / sqrtf(sigma_data * sigma_data + sg * sg);
  }
  const long long row_base = (long long)cloud * rows_per_cloud;
  for (int cq = threadIdx.x; cq < C / 4; cq += blockDim.x) {
    float wv[4][3], bv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int c = cq * 4 + j;
      wv[j][0] = __ldg(w + c * 3 + 0);
      wv[j][1] = __ldg(w + c * 3 + 1);
      wv[j][2] = __ldg(w + c * 3 + 2);
      bv[j] = __ldg(b + c);
    }
    float s1[4] = {0, 0, 0, 0}, s2[4] = {0, 0, 0, 0};
    for (int r = r0; r < r1; ++r) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      if (r < valid_rows) {
        const float* g = xin + ((long long)cloud * valid_rows + r) * 3;
        const float g0 = c_in * __ldg(g), g1 = c_in * __ldg(g + 1), g2 = c_in * __ldg(g + 2);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          o[j] = bv[j] + g0 * wv[j][0] + g1 * wv[j][1] + g2 * wv[j][2];
          s1[j] += o[j];
          s2[j] += o[j] * o[j];
        }
      }
      *reinterpret_cast<float4*>(x + (row_base + r) * ldx + cq * 4) = make_float4(o[0], o[1], o[2], o[3]);
      if (xb != nullptr)
        *reinterpret_cast<uint2*>(xb + (row_base + r) * ldxb + cq * 4) = make_uint2(pack_bf16x2(o[0], o[1]), pack_bf16x2(o[2], o[3]));
    }
    if (stats != nullptr) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int g = (cq * 4 + j) / gs;
        atomicAdd(&sgrp[g * 2], static_cast<double>(s1[j]));
        atomicAdd(&sgrp[g * 2 + 1], static_cast<double>(s2[j]));
      }
    }
  }
  if (stats != nullptr) {
    __syncthreads();
    for (int i = threadIdx.x; i < ngroups * 2; i += blockDim.x)
      atomicAdd(stats + (long long)cloud * ngroups * 2 + i, sgrp[i]);
  }
}

// ------------------------------------------------------------------------------------------------
// Output head + EDM preconditioning + sampler update, one warp per point.
//   F = W_out . norm(x_row) + b_out           (models/ray.py:56-59,120 / models/linear_lift.py:26-29,46)
//   D = c_skip * xin + c_out * F              (diffusion.py:46-57)
//   mode 2: Euler step, mode 3: Heun correction + churn of the next step (diffusion.py:317-347)
constexpr int HEAD_WARPS = 8;
constexpr int HEAD_ROWS_PER_WARP = 32;  // 256 rows per block: the per-block weight folding is amortised
constexpr int HEAD_MAX_NQ = 8;  // C <= 1024

// EDM preconditioning + sampler update of one output element (lanes 0..2 of the warp that owns the row).
__device__ __forceinline__ void head_finish(const gecco_head_args& a, long long idx, float F, float c_skip, float c_out) {
  if (a.mode == 0) {
    a.out_f32[idx] = F;
    return;
  }
  const float xi = a.xin[idx];
  const float D = c_skip * xi + c_out * F;
  if (a.mode == 1) {
    a.out_f32[idx] = D;
  } else if (a.mode == 2) {  // Euler
    const double xh = a.x_hat[idx];
    const double d_cur = (xh - static_cast<double>(D)) / a.t_hat;
    const double xn = xh + (a.t_next - a.t_hat) * d_cur;
    a.d_cur[idx] = d_cur;
    a.x_next[idx] = xn;
    a.xin_next[idx] = static_cast<float>(xn);
  } else {  // Heun correction, then churn for the next step
    const double xh = a.x_hat[idx];
    const double xn = a.x_next[idx];
    const double d_prime = (xn - static_cast<double>(D)) / a.t_next;
    double xnew = xh + (a.t_next - a.t_hat) * (0.5 * a.d_cur[idx] + 0.5 * d_prime);
    // the reference multiplies the 0-dim float64 churn factor into the fp32 noise tensor, which torch
    // evaluates in fp32 (diffusion.py:325)
    if (a.noise_next != nullptr)
      xnew = xnew + static_cast<double>(__fmul_rn(static_cast<float>(a.churn_next), a.noise_next[idx]));
    a.x_hat[idx] = xnew;
    a.xin_next[idx] = static_cast<float>(xnew);
  }
}

// NQ = C / 128 float4 per lane.  The normalisation is folded into the three weight rows once per block:
//   GroupNorm:  F_o = sum_c x_c (r_c w_oc) - sum_c m_c r_c w_oc + b_o        (statistics per cloud)
//   LayerNorm:  F_o = rstd (sum_c x_c w_oc - mean sum_c w_oc) + b_o          (statistics per row)
// so a row costs NQ 16-byte loads, 12 NQ FMAs and three warp reductions; every warp keeps two rows in flight.
template <int NQ>
__global__ void __launch_bounds__(HEAD_WARPS * 32)
head_kernel(const gecco_head_args a) {
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  extern __shared__ float smem_head[];  // [groups][2] mean, rstd (GroupNorm mode)
  const int cloud = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int C = NQ * 128;
  const int gs = (a.norm == 2) ? C / a.groups : 1;
  if (a.norm == 2) {
    const double count = static_cast<double>(a.valid_rows) * gs;
    const double* cstats = a.stats + (long long)cloud * (C / a.stat_gs) * 2;
    for (int g = threadIdx.x; g < a.groups; g += blockDim.x) {
      float mean, rstd;
      group_mean_rstd(cstats, g, gs, a.stat_gs, count, a.eps, mean, rstd);
      smem_head[g * 2] = mean;
      smem_head[g * 2 + 1] = rstd;
    }
    __syncthreads();
  }
  const float sg = a.sigma != nullptr ? __ldg(a.sigma + (long long)cloud * a.sigma_stride) : 0.f;
  const float sd = a.sigma_data;
  const float c_skip = sd * sd / (sg * sg + sd * sd);
  const float c_out = sg * sd / sqrtf(sg * sg + sd * sd);

  // this lane's slice of the three (normalisation-folded) weight rows and the per-cloud constants
  float4 w[3][NQ];
  float kc[3];  // GroupNorm: sum_c m_c r_c w_oc;  LayerNorm: sum_c w_oc
#pragma unroll
  for (int o = 0; o < 3; ++o) {
    float acc = 0.f;
#pragma unroll
    for (int i = 0; i < NQ; ++i) {
      float4 w4 = __ldg(reinterpret_cast<const float4*>(a.w_out + (long long)o * C + i * 128 + lane * 4));
      if (a.norm == 2) {
        const int c = i * 128 + lane * 4;
        float m[4], r[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) { m[j] = smem_head[((c + j) / gs) * 2]; r[j] = smem_head[((c + j) / gs) * 2 + 1]; }
        w4.x *= r[0]; w4.y *= r[1]; w4.z *= r[2]; w4.w *= r[3];
        acc += m[0] * w4.x + m[1] * w4.y + m[2] * w4.z + m[3] * w4.w;
      } else {
        acc += w4.x + w4.y + w4.z + w4.w;
      }
      w[o][i] = w4;
    }
    kc[o] = warp_sum(acc);
  }
  const float bo = lane < 3 ? __ldg(a.b_out + lane) : 0.f;

  const int rb = (blockIdx.x * HEAD_WARPS + warp) * HEAD_ROWS_PER_WARP;
  const float* xc = a.x + (long long)cloud * a.rows_per_cloud * a.ldx + lane * 4;
  if (a.norm != 1) {
    // four rows in flight; the twelve dot products are reduced together (reduce-scatter: 16 shuffles for four rows,
    // the sum of value j lands in lanes 2 j and 2 j + 1) and lanes 8 u + 2 o finish output o of row u
#pragma unroll 1
    for (int rr = 0; rr < HEAD_ROWS_PER_WARP; rr += 4) {
      const int r0 = rb + rr;
      if (r0 >= a.valid_rows) break;
      float4 v[4][NQ];
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int i = 0; i < NQ; ++i)
          v[u][i] = r0 + u < a.valid_rows ? __ldg(reinterpret_cast<const float4*>(xc + (long long)(r0 + u) * a.ldx + i * 128))
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
      float f[16];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
#pragma unroll
        for (int o = 0; o < 3; ++o) {
          float acc = 0.f;
#pragma unroll
          for (int i = 0; i < NQ; ++i)
            acc += v[u][i].x * w[o][i].x + v[u][i].y * w[o][i].y + v[u][i].z * w[o][i].z + v[u][i].w * w[o][i].w;
          f[4 * u + o] = acc;
        }
        f[4 * u + 3] = 0.f;
      }
#pragma unroll
      for (int half = 8; half >= 1; half >>= 1) {
        const int off = 2 * half;
        const bool upper = (lane & off) != 0;
#pragma unroll
        for (int i = 0; i < half; ++i) {
          const float send = upper ? f[i] : f[i + half];
          const float keep = upper ? f[i + half] : f[i];
          f[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
        }
      }
      const float tot = f[0] + __shfl_xor_sync(0xffffffffu, f[0], 1);
      const int u = lane >> 3, o = (lane >> 1) & 3;
      if ((lane & 1) == 0 && o < 3 && r0 + u < a.valid_rows) {
        const float k = o == 0 ? kc[0] : (o == 1 ? kc[1] : kc[2]);
        const float F = tot - (a.norm == 2 ? k : 0.f) + __ldg(a.b_out + o);
        head_finish(a, ((long long)cloud * a.valid_rows + r0 + u) * 3 + o, F, c_skip, c_out);
      }
    }
    return;
  }
#pragma unroll 1
  for (int rr = 0; rr < HEAD_ROWS_PER_WARP; rr += 2) {
    const int r0 = rb + rr;
    if (r0 >= a.valid_rows) break;
    const bool two = r0 + 1 < a.valid_rows;
    float4 v[2][NQ];
#pragma unroll
    for (int i = 0; i < NQ; ++i) {
      v[0][i] = __ldg(reinterpret_cast<const float4*>(xc + (long long)r0 * a.ldx + i * 128));
      v[1][i] = two ? __ldg(reinterpret_cast<const float4*>(xc + (long long)(r0 + 1) * a.ldx + i * 128)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (u == 1 && !two) break;
      float f[3];
#pragma unroll
      for (int o = 0; o < 3; ++o) {
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < NQ; ++i)
          acc += v[u][i].x * w[o][i].x + v[u][i].y * w[o][i].y + v[u][i].z * w[o][i].z + v[u][i].w * w[o][i].w;
        f[o] = warp_sum(acc);
      }
      if (a.norm == 1) {  // LayerNorm over channels, no affine: statistics of this row
        float s = 0.f;
#pragma unroll
        for (int i = 0; i < NQ; ++i) s += v[u][i].x + v[u][i].y + v[u][i].z + v[u][i].w;
        const float mean = warp_sum(s) / C;
        float q = 0.f;
#pragma unroll
        for (int i = 0; i < NQ; ++i) {
          const float d0 = v[u][i].x - mean, d1 = v[u][i].y - mean, d2 = v[u][i].z - mean, d3 = v[u][i].w - mean;
          q += d0 * d0 + d1 * d1 + d2 * d2 + d3 * d3;
        }
        const float rstd = rsqrtf(warp_sum(q) / C + a.eps);
#pragma unroll
        for (int o = 0; o < 3; ++o) f[o] = rstd * (f[o] - mean * kc[o]);
      } else if (a.norm == 2) {
#pragma unroll
        for (int o = 0; o < 3; ++o) f[o] -= kc[o];
      }
      if (lane < 3) {
        const float F = (lane == 0 ? f[0] : (lane == 1 ? f[1] : f[2])) + bo;
        head_finish(a, ((long long)cloud * a.valid_rows + r0 + u) * 3 + lane, F, c_skip, c_out);
      }
    }
  }
}

// x_hat = scale0 * latents (+ churn * noise); also the fp32 network input.  (diffusion.py:308,323-325)
__global__ void sampler_init_kernel(const float* __restrict__ latents, const float* __restrict__ noise, double t0,
                                    double churn, long long n, double* __restrict__ x_hat, float* __restrict__ xin) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double x = static_cast<double>(latents[i]) * t0;
  if (noise != nullptr) x = x + static_cast<double>(__fmul_rn(static_cast<float>(churn), noise[i]));  // fp32 product, see head_kernel
  x_hat[i] = x;
  xin[i] = static_cast<float>(x);
}

// ------------------------------------------------------------------------------------------------
// Reparametrisations (reparam.py).  T = float or double.
template <typename T>
struct RP {
  T mean[3], sigma[3];
  T logit_scale;
};

template <typename T>
__device__ __forceinline__ void project_pt(const T* p, const T* K, T& u, T& v) {
  // kornia project_points: scale = |z| > 1e-8 ? 1/(z + 1e-8) : 1
  const T z = p[2];
  const T sc = (fabs(z) > T(1e-8)) ? T(1) / (z + T(1e-8)) : T(1);
  u = p[0] * sc * K[0] + K[2];
  v = p[1] * sc * K[4] + K[5];
}

template <typename T>
__global__ void reparam_kernel(const T* __restrict__ in, T* __restrict__ out, const float* __restrict__ Kmat,
                               int kind, int to_data, RP<T> rp, int points_per_cloud, long long n_points) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_points) return;
  T p[3] = {in[i * 3], in[i * 3 + 1], in[i * 3 + 2]};
  T o[3];
  if (kind == 1) {  // GaussianReparam, reparam.py:58-64
    for (int j = 0; j < 3; ++j) o[j] = to_data ? p[j] * rp.sigma[j] + rp.mean[j] : (p[j] - rp.mean[j]) / rp.sigma[j];
  } else if (kind == 2) {  // UVLReparam, reparam.py:122-201
    T K[9];
    const float* Kc = Kmat + (i / points_per_cloud) * 9;
    for (int j = 0; j < 9; ++j) K[j] = static_cast<T>(Kc[j]);
    if (to_data) {
      T uvl[3];
      for (int j = 0; j < 3; ++j) uvl[j] = p[j] * rp.sigma[j] + rp.mean[j];
      const T h = (tanh(uvl[0]) * rp.logit_scale + T(1)) / T(2);
      const T w = (tanh(uvl[1]) * rp.logit_scale + T(1)) / T(2);
      const T d = exp(uvl[2]);
      const T x = (h - K[2]) / K[0];
      const T y = (w - K[5]) / K[4];
      T nrm = sqrt(x * x + y * y + T(1));
      nrm = nrm > T(1e-12) ? nrm : T(1e-12);
      o[0] = x / nrm * d;
      o[1] = y / nrm * d;
      o[2] = T(1) / nrm * d;
    } else {
      T u, v;
      project_pt(p, K, u, v);
      const T d = sqrt(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
      const T r0 = atanh((T(2) * u - T(1)) / rp.logit_scale);
      const T r1 = atanh((T(2) * v - T(1)) / rp.logit_scale);
      const T r2 = log(d);
      o[0] = (r0 - rp.mean[0]) / rp.sigma[0];
      o[1] = (r1 - rp.mean[1]) / rp.sigma[1];
      o[2] = (r2 - rp.mean[2]) / rp.sigma[2];
    }
  } else {
    for (int j = 0; j < 3; ++j) o[j] = p[j];
  }
  out[i * 3] = o[0];
  out[i * 3 + 1] = o[1];
  out[i * 3 + 2] = o[2];
}

}  // namespace

// ---------------------------------------------------------------- host launchers (used by engine.cu too)
int launch_group_stats(const float* x, long long ldx, int clouds, int rows_per_cloud, int valid_rows, int C, int gs,
                       double* stats, cudaStream_t s) {
  GECCO_REQUIRE(C % 4 == 0 && gs > 0 && C % gs == 0, "group_stats: bad channel layout C=%d gs=%d", C, gs);
  GECCO_REQUIRE(ldx % 4 == 0, "group_stats: ldx must be a multiple of 4");
  dim3 grid(ceil_div(valid_rows, STAT_ROWS), clouds);
  const int threads = C / 4 < 256 ? ((C / 4 + 31) / 32) * 32 : 256;
  group_stats_kernel<<<grid, threads, (C / gs) * 2 * sizeof(double), s>>>(x, ldx, rows_per_cloud, valid_rows, C, gs, stats);
  GECCO_CHECK_LAUNCH("group_stats_kernel");
  return GECCO_OK;
}

int launch_adagn(const gecco_adagn_args& a, cudaStream_t s) {
  GECCO_REQUIRE(a.c % 4 == 0 && a.groups > 0 && a.c % a.groups == 0, "adagn: bad channel layout");
  GECCO_REQUIRE(a.stat_gs > 0 && (a.c / a.groups) % a.stat_gs == 0, "adagn: group size %d is not a multiple of the statistics granularity %d",
                a.c / a.groups, a.stat_gs);
  GECCO_REQUIRE(a.out_bf16 || a.out_f32, "adagn: no output");
  GECCO_REQUIRE(a.ldx % 4 == 0 && (!a.out_bf16 || a.ldo16 % 4 == 0) && (!a.out_f32 || a.ldo32 % 4 == 0), "adagn: bad leading dimension");
  dim3 grid(ceil_div(a.rows_per_cloud, ADAGN_ROWS), a.clouds);
  const int threads = a.c / 4 < 256 ? ((a.c / 4 + 31) / 32) * 32 : 256;
  launch_small(adagn_apply_kernel, grid, dim3(threads), 0, s, a.x, a.ldx, a.stats, a.stat_gs, a.t, a.t_stride, a.ctx_dim, a.scale_w,
               a.scale_b, a.bias_w, a.bias_b, a.rows_per_cloud, a.valid_rows, a.c, a.groups, a.eps,
               static_cast<__nv_bfloat16*>(a.out_bf16), a.ldo16, a.out_f32, a.ldo32);
  GECCO_CHECK_LAUNCH("adagn_apply_kernel");
  return GECCO_OK;
}

int launch_fold_adagn(const gecco_fold_adagn_args& a, cudaStream_t s) {
  GECCO_REQUIRE(a.w && a.stats && a.t && a.w_folded_bf16 && a.bias_folded, "fold_adagn: null argument");
  GECCO_REQUIRE(a.c % 4 == 0 && a.c <= FOLD_MAXC && a.ldw % 4 == 0 && a.ldwf % 4 == 0, "fold_adagn: C must be a multiple of 4 (<= %d)", FOLD_MAXC);
  GECCO_REQUIRE(a.groups > 0 && a.c % a.groups == 0 && a.stat_gs > 0 && (a.c / a.groups) % a.stat_gs == 0,
                "fold_adagn: group size must be a multiple of the statistics granularity");
  GECCO_REQUIRE(a.ctx_dim == 1, "fold_adagn: t_embed_dim must be 1");
  GECCO_REQUIRE(a.groups <= 128, "fold_adagn: at most 128 groups");
  if (a.n_out == 0 || a.clouds == 0) return GECCO_OK;
  dim3 grid(ceil_div(a.n_out, FOLD_ROWS), ceil_div(a.clouds, FOLD_CLOUDS));
  const size_t smem = (size_t)FOLD_CLOUDS * (2 * a.c + 2 * a.groups) * sizeof(float);
  const char* ffv = getenv("GECCO_FOLD_FAST");  // GECCO_FOLD_FAST=0: the generic kernel (A/B measurements, tests)
  const bool fast_ok = !(ffv != nullptr && ffv[0] == '0');
  if (fast_ok && a.c == 384) {
    launch_small(fold_adagn_fast_kernel<3>, grid, dim3(FOLD_THREADS), smem, s, a.w, a.ldw, a.bias, a.n_out, a.stats, a.stat_gs, a.groups,
                 (double)a.valid_rows * (a.c / a.groups), a.eps, a.t, a.t_stride, a.scale_w, a.scale_b, a.bias_w, a.bias_b,
                 a.clouds, static_cast<__nv_bfloat16*>(a.w_folded_bf16), a.ldwf, a.wf_cloud_stride, a.bias_folded, a.bias_stride);
    GECCO_CHECK_LAUNCH("fold_adagn_fast_kernel");
    return GECCO_OK;
  }
  launch_small(fold_adagn_kernel, grid, dim3(FOLD_THREADS), smem, s, a.w, a.ldw, a.bias, a.n_out, a.c, a.stats, a.stat_gs, a.groups,
               (double)a.valid_rows * (a.c / a.groups), a.eps, a.t, a.t_stride, a.scale_w, a.scale_b, a.bias_w, a.bias_b,
               a.clouds, static_cast<__nv_bfloat16*>(a.w_folded_bf16), a.ldwf, a.wf_cloud_stride, a.bias_folded, a.bias_stride);
  GECCO_CHECK_LAUNCH("fold_adagn_kernel");
  return GECCO_OK;
}

int launch_lift(const gecco_lift_args& a, cudaStream_t s) {
  GECCO_REQUIRE(a.c % 4 == 0 && a.ldx % 4 == 0, "lift: bad channel layout");
  GECCO_REQUIRE(!a.x_bf16 || a.ldxb % 4 == 0, "lift: bf16 leading dimension must be a multiple of 4");
  GECCO_REQUIRE(!a.stats || (a.stat_gs > 0 && a.c % a.stat_gs == 0), "lift: bad statistics granularity");
  dim3 grid(ceil_div(a.rows_per_cloud, LIFT_ROWS), a.clouds);
  const int threads = a.c / 4 < 256 ? ((a.c / 4 + 31) / 32) * 32 : 256;
  const int gs = a.stats ? a.stat_gs : a.c;
  lift_kernel<<<grid, threads, (a.c / gs) * 2 * sizeof(double), s>>>(a.xin, a.sigma, a.sigma_stride, a.sigma_data, a.w, a.b,
                                                                   a.rows_per_cloud, a.valid_rows, a.c, gs, a.x, a.ldx,
                                                                   static_cast<__nv_bfloat16*>(a.x_bf16), a.ldxb, a.stats);
  GECCO_CHECK_LAUNCH("lift_kernel");
  return GECCO_OK;
}

int launch_head(const gecco_head_args& a, cudaStream_t s) {
  GECCO_REQUIRE(a.c % 128 == 0 && a.c <= 128 * HEAD_MAX_NQ, "head: C must be a multiple of 128 and <= 1024");
  GECCO_REQUIRE(a.ldx % 4 == 0, "head: ldx must be a multiple of 4");
  GECCO_REQUIRE(a.norm != 2 || (a.stats && a.groups > 0 && a.c % a.groups == 0 && (a.c / a.groups) % a.stat_gs == 0),
                "head: GroupNorm needs statistics with a granularity dividing the group size");
  GECCO_REQUIRE(a.mode >= 0 && a.mode <= 3, "head: bad mode");
  GECCO_REQUIRE(a.mode == 0 || (a.xin && a.sigma), "head: preconditioning needs xin and sigma");
  GECCO_REQUIRE(a.mode > 1 || a.out_f32, "head: no output");
  GECCO_REQUIRE(a.mode < 2 || (a.x_hat && a.x_next && a.d_cur && a.xin_next), "head: sampler state missing");
  dim3 grid(ceil_div(a.valid_rows, HEAD_WARPS * HEAD_ROWS_PER_WARP), a.clouds);
  const size_t sm = a.norm == 2 ? a.groups * 2 * sizeof(float) : 0;
  switch (a.c / 128) {
#define GECCO_HEAD_CASE(NQ) case NQ: launch_small(head_kernel<NQ>, grid, dim3(HEAD_WARPS * 32), sm, s, a); break;
    GECCO_HEAD_CASE(1) GECCO_HEAD_CASE(2) GECCO_HEAD_CASE(3) GECCO_HEAD_CASE(4)
    GECCO_HEAD_CASE(5) GECCO_HEAD_CASE(6) GECCO_HEAD_CASE(7) GECCO_HEAD_CASE(8)
#undef GECCO_HEAD_CASE
    default: GECCO_REQUIRE(false, "head: C must be a multiple of 128 and <= 1024");
  }
  GECCO_CHECK_LAUNCH("head_kernel");
  return GECCO_OK;
}

// Upsampling helpers (diffusion.py:430-437, 447-449, 464-466).  torch evaluates `0-dim float64 * float32 tensor` in fp32,
// so the noise products are fp32 and only the accumulation into the sampler state is float64.
__global__ void seed_renoise_kernel(const float* __restrict__ data, const float* __restrict__ noise, float t, long long n,
                                    float* __restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = __fadd_rn(data[i], __fmul_rn(noise[i], t));  // data + randn * t_cur, two roundings like torch
}
// x_hat = (src [+ c1 * n1]) + c2 * n2: re-noising of the previous sub-step (optional) followed by the churn of this one.
__global__ void substep_noise_kernel(const double* __restrict__ src, const float* __restrict__ n1, float c1,
                                     const float* __restrict__ n2, float c2, long long n, double* __restrict__ x_hat,
                                     float* __restrict__ xin) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double x = src[i];
  if (n1 != nullptr) x = x + static_cast<double>(__fmul_rn(c1, n1[i]));
  if (n2 != nullptr) x = x + static_cast<double>(__fmul_rn(c2, n2[i]));
  x_hat[i] = x;
  xin[i] = static_cast<float>(x);
}

int launch_seed_renoise(const float* data, const float* noise, float t, long long n, float* out, cudaStream_t s) {
  seed_renoise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(data, noise, t, n, out);
  GECCO_CHECK_LAUNCH("seed_renoise_kernel");
  return GECCO_OK;
}
int launch_substep_noise(const double* src, const float* n1, float c1, const float* n2, float c2, long long n, double* x_hat,
                         float* xin, cudaStream_t s) {
  substep_noise_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(src, n1, c1, n2, c2, n, x_hat, xin);
  GECCO_CHECK_LAUNCH("substep_noise_kernel");
  return GECCO_OK;
}

int launch_sampler_init(const float* latents, const float* noise, double t0, double churn, long long n, double* x_hat,
                        float* xin, cudaStream_t s) {
  sampler_init_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(latents, noise, t0, churn, n, x_hat, xin);
  GECCO_CHECK_LAUNCH("sampler_init_kernel");
  return GECCO_OK;
}

}  // namespace gecco

extern "C" int gecco_group_stats(const float* x, int64_t ldx, int32_t clouds, int32_t rows_per_cloud, int32_t valid_rows,
                                 int32_t c, int32_t group_size, double* stats, void* stream) {
  return gecco::launch_group_stats(x, ldx, clouds, rows_per_cloud, valid_rows, c, group_size, stats,
                                   static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_adagn(const gecco_adagn_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_adagn: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_adagn(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_fold_adagn(const gecco_fold_adagn_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_fold_adagn: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_fold_adagn(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_lift(const gecco_lift_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_lift: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_lift(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_head(const gecco_head_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_head: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_head(*a, static_cast<cudaStream_t>(stream));
}

namespace gecco {
namespace {
// GaussianActivation (models/activation.py:17-24) as a stand-alone op: y = exp(-x^2 / (2 alpha^2)), optionally
// (y - 0.7) / 0.28.  On the hot path the activation lives in the epilogue of the GEMM that produces x.
__global__ void gaussian_act_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, float k, int normalized) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    const float4 v = *reinterpret_cast<const float4*>(x + i);
    float4 o;
    o.x = exp2f(v.x * v.x * k); o.y = exp2f(v.y * v.y * k); o.z = exp2f(v.z * v.z * k); o.w = exp2f(v.w * v.w * k);
    if (normalized) { o.x = (o.x - 0.7f) / 0.28f; o.y = (o.y - 0.7f) / 0.28f; o.z = (o.z - 0.7f) / 0.28f; o.w = (o.w - 0.7f) / 0.28f; }
    *reinterpret_cast<float4*>(y + i) = o;
  } else {
    for (long long j = i; j < n; ++j) {
      float o = exp2f(x[j] * x[j] * k);
      y[j] = normalized ? (o - 0.7f) / 0.28f : o;
    }
  }
}
}  // namespace
}  // namespace gecco

extern "C" int gecco_gaussian_activation(const float* x, float* y, int64_t n, float alpha, int32_t normalized, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(x != nullptr && y != nullptr && n >= 0, "gaussian_activation: null argument");
  GECCO_REQUIRE(alpha != 0.f, "gaussian_activation: alpha must be non-zero");
  GECCO_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0,
                "gaussian_activation: buffers must be 16-byte aligned");
  if (n == 0) return GECCO_OK;
  const float k = static_cast<float>(-1.4426950408889634 / (2.0 * (double)alpha * (double)alpha));
  const long long quads = (n + 3) / 4;
  gaussian_act_kernel<<<(unsigned)((quads + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(x, y, n, k, normalized);
  GECCO_CHECK_LAUNCH("gaussian_act_kernel");
  return GECCO_OK;
}

extern "C" int gecco_reparam(const void* in, void* out, int32_t is_double, int32_t kind, int32_t to_data,
                             const float* mean, const float* sigma, float logit_scale, const float* K,
                             int32_t clouds, int32_t points_per_cloud, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(kind >= 0 && kind <= 2, "reparam: unknown kind %d", kind);
  GECCO_REQUIRE(kind != 2 || K != nullptr, "reparam: UVL needs the camera matrices");
  const long long n = (long long)clouds * points_per_cloud;
  if (n == 0) return GECCO_OK;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const unsigned blocks = (unsigned)((n + 255) / 256);
  if (is_double) {
    RP<double> rp;
    for (int j = 0; j < 3; ++j) { rp.mean[j] = mean ? mean[j] : 0.0; rp.sigma[j] = sigma ? sigma[j] : 1.0; }
    rp.logit_scale = logit_scale;
    reparam_kernel<double><<<blocks, 256, 0, s>>>(static_cast<const double*>(in), static_cast<double*>(out), K, kind,
                                                  to_data, rp, points_per_cloud, n);
  } else {
    RP<float> rp;
    for (int j = 0; j < 3; ++j) { rp.mean[j] = mean ? mean[j] : 0.f; rp.sigma[j] = sigma ? sigma[j] : 1.f; }
    rp.logit_scale = logit_scale;
    reparam_kernel<float><<<blocks, 256, 0, s>>>(static_cast<const float*>(in), static_cast<float*>(out), K, kind,
                                                 to_data, rp, points_per_cloud, n);
  }
  GECCO_CHECK_LAUNCH("reparam_kernel");
  return GECCO_OK;
}
