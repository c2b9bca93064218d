// Projective feature lookup (models/ray.py:64-87): reparametrise the EDM-scaled points to data
// space, project them through the camera, bilinearly gather every level of the channels-last
// feature pyramid.  One warp per point; a lane owns fixed 8-channel chunks (one 16 B load per tap),
// so the [points, sum C] output row is written with fully coalesced 16 B stores and the GroupNorm
// statistics of models/ray.py:53 are accumulated per lane and reduced once per CTA.
// Also: folding of that GroupNorm into per-cloud projection weights, and the NCHW fp32 ->
// NHWC bf16 repack of the pyramid.
#include "common.cuh"
#include "ptx.cuh"

#include <stdlib.h>

namespace gecco {

namespace {

constexpr int LK_WARPS = 8;
constexpr int LK_MAXCH = 4;          // 8-channel chunks per lane -> up to 1024 channels
constexpr int LK_POINTS_PER_WARP = 16;

struct LookupP {
  const float* xin;
  const float* sigma;
  int sigma_stride;
  float sigma_data;
  int reparam;
  float mean[3], rsig[3], logit_scale;
  const float* K;
  int n_levels;
  const __nv_bfloat16* lvl_ptr[GECCO_MAX_LEVELS];
  int lvl_h[GECCO_MAX_LEVELS], lvl_w[GECCO_MAX_LEVELS], lvl_c[GECCO_MAX_LEVELS];
  int points, rows_per_cloud, ctot;
  __nv_bfloat16* out16;
  long long ldo16;
  float* out32;
  long long ldo32;
  double* stats;
  int stat_groups;
  int glob_mask;  // staged kernel, HYBRID: bit l set = level l is NOT staged, its taps are gathered from global memory (L2)
};

__device__ __forceinline__ void bf16x8_to_float(const uint4& q, float* f) {
  const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&q);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 t = __bfloat1622float2(h[i]);
    f[2 * i] = t.x;
    f[2 * i + 1] = t.y;
  }
}

// Data-space point -> normalised image coordinates (reparam.diffusion_to_data + kornia project_points), then the
// grid_sample grid value 2 uv - 1 (models/ray.py:71-82).
__device__ __forceinline__ void lookup_coords(const LookupP& p, const float (&xyz)[3], float c_in, float fx, float cx,
                                              float fy, float cy, float& gx, float& gy) {
  float g[3] = {c_in * xyz[0], c_in * xyz[1], c_in * xyz[2]};
  float d[3];
  if (p.reparam == 1) {  // GaussianReparam.diffusion_to_data (reparam.py:62-64)
    for (int j = 0; j < 3; ++j) d[j] = g[j] * p.rsig[j] + p.mean[j];
  } else if (p.reparam == 2) {  // UVLReparam.diffusion_to_data (reparam.py:166-201)
    const float u0 = g[0] * p.rsig[0] + p.mean[0];
    const float v0 = g[1] * p.rsig[1] + p.mean[1];
    const float l0 = g[2] * p.rsig[2] + p.mean[2];
    const float h = (tanhf(u0) * p.logit_scale + 1.0f) / 2.0f;
    const float w = (tanhf(v0) * p.logit_scale + 1.0f) / 2.0f;
    const float dep = expf(l0);
    const float x = (h - cx) / fx, y = (w - cy) / fy;
    float nrm = sqrtf(x * x + y * y + 1.0f);
    nrm = fmaxf(nrm, 1e-12f);
    d[0] = x / nrm * dep;
    d[1] = y / nrm * dep;
    d[2] = 1.0f / nrm * dep;
  } else {
    for (int j = 0; j < 3; ++j) d[j] = g[j];
  }
  // kornia project_points (models/ray.py:74)
  const float z = d[2];
  const float sc = (fabsf(z) > 1e-8f) ? 1.0f / (z + 1e-8f) : 1.0f;
  const float u = d[0] * sc * fx + cx;
  const float v = d[1] * sc * fy + cy;
  gx = u * 2.0f - 1.0f;
  gy = v * 2.0f - 1.0f;
}

// Bilinear tap geometry of one level (F.grid_sample, zeros padding, align_corners=False): pixel index y * W + x and
// weight of the four taps.  A tap outside the map contributes 0: its weight is zeroed and its index is 0
// (non-finite coordinates give NaN weights, which the validity test turns into zeros exactly like grid_sample's
// padding).
__device__ __forceinline__ void lookup_geom(int H, int W, float gx, float gy, int (&pix)[4], float (&w)[4], bool (&tv)[4]) {
  const float ix = ((gx + 1.0f) * W - 1.0f) / 2.0f;
  const float iy = ((gy + 1.0f) * H - 1.0f) / 2.0f;
  const float x0 = floorf(ix), y0 = floorf(iy);
  const float x1 = x0 + 1.0f, y1 = y0 + 1.0f;
  const bool vx0 = x0 >= 0.f && x0 <= (float)(W - 1), vx1 = x1 >= 0.f && x1 <= (float)(W - 1);
  const bool vy0 = y0 >= 0.f && y0 <= (float)(H - 1), vy1 = y1 >= 0.f && y1 <= (float)(H - 1);
  const int xi0 = vx0 ? (int)x0 : 0, xi1 = vx1 ? (int)x1 : 0, yi0 = vy0 ? (int)y0 : 0, yi1 = vy1 ? (int)y1 : 0;
  tv[0] = vx0 && vy0; tv[1] = vx1 && vy0; tv[2] = vx0 && vy1; tv[3] = vx1 && vy1;
  pix[0] = yi0 * W + xi0; pix[1] = yi0 * W + xi1; pix[2] = yi1 * W + xi0; pix[3] = yi1 * W + xi1;
  w[0] = tv[0] ? (x1 - ix) * (y1 - iy) : 0.f;
  w[1] = tv[1] ? (ix - x0) * (y1 - iy) : 0.f;
  w[2] = tv[2] ? (x1 - ix) * (iy - y0) : 0.f;
  w[3] = tv[3] ? (ix - x0) * (iy - y0) : 0.f;
}

// The four bilinear taps of one 8-channel chunk: issue the loads.
struct Taps {
  uint4 q[4];
  float w[4];
};
__device__ __forceinline__ void lookup_issue(const __nv_bfloat16* __restrict__ base, int H, int W, int C, float gx, float gy,
                                             Taps& t) {
  int pix[4];
  bool tv[4];
  lookup_geom(H, W, gx, gy, pix, t.w, tv);
#pragma unroll
  for (int i = 0; i < 4; ++i) t.q[i] = tv[i] ? __ldg(reinterpret_cast<const uint4*>(base + pix[i] * C)) : make_uint4(0, 0, 0, 0);
}
__device__ __forceinline__ void lookup_blend(const Taps& t, float (&acc)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float f[8];
    bf16x8_to_float(t.q[i], f);
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = fmaf(f[j], t.w[i], acc[j]);
  }
}

// NCH: 8-channel chunks per lane (ceil(sum C / 256)).  Two points of a warp are in flight together (2 x NCH x 4
// independent 16 B gathers per lane) because the kernel is bound by the latency of the L2-resident gathers.
template <int NCH>
__global__ void __launch_bounds__(LK_WARPS * 32, 2) lookup_kernel(const LookupP p) {
  extern __shared__ double sgrp[];  // [stat_groups][2]; double: order-independent partial sums
  const int cloud = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (p.stats != nullptr) {
    for (int i = threadIdx.x; i < p.stat_groups * 2; i += blockDim.x) sgrp[i] = 0.0;
    __syncthreads();
  }
  // fixed chunk -> (level, channel) assignment of this lane
  const __nv_bfloat16* ch_ptr[NCH];
  int ch_h[NCH], ch_w[NCH], ch_c[NCH], ch_col[NCH];
  // statistics: a chunk of 8 channels touches at most two GroupNorm groups (group size >= 8): channels [0, bnd) belong to
  // group gA, channels [bnd, 8) to group gA + 1
  int bnd[NCH], gA[NCH];
  const int gsz = p.stats != nullptr ? p.ctot / p.stat_groups : 8;
#pragma unroll
  for (int k = 0; k < NCH; ++k) {
    const int col = (lane + 32 * k) * 8;
    ch_col[k] = col;
    ch_ptr[k] = nullptr;
    ch_h[k] = ch_w[k] = ch_c[k] = 0;
    int off = 0;
    for (int l = 0; l < p.n_levels; ++l) {
      if (col >= off && col < off + p.lvl_c[l]) {
        ch_h[k] = p.lvl_h[l];
        ch_w[k] = p.lvl_w[l];
        ch_c[k] = p.lvl_c[l];
        ch_ptr[k] = p.lvl_ptr[l] + (long long)cloud * p.lvl_h[l] * p.lvl_w[l] * p.lvl_c[l] + (col - off);
      }
      off += p.lvl_c[l];
    }
    gA[k] = col / gsz;
    const int next = (gA[k] + 1) * gsz - col;  // channels of this chunk that still belong to group gA
    bnd[k] = next < 8 ? next : 8;
  }
  float sA1[NCH], sA2[NCH], sB1[NCH], sB2[NCH];
#pragma unroll
  for (int k = 0; k < NCH; ++k) sA1[k] = sA2[k] = sB1[k] = sB2[k] = 0.f;

  float c_in = 1.f;
  if (p.sigma != nullptr) {
    const float sg = __ldg(p.sigma + (long long)cloud * p.sigma_stride);
    c_in = 1.0f / sqrtf(p.sigma_data * p.sigma_data + sg * sg);
  }
  const float* Kc = p.K + (long long)cloud * 9;
  const float fx = __ldg(Kc + 0), cx = __ldg(Kc + 2), fy = __ldg(Kc + 4), cy = __ldg(Kc + 5);

  const int stride = gridDim.x * LK_WARPS;
  for (int pt = blockIdx.x * LK_WARPS + warp; pt < p.points; pt += 2 * stride) {
    const int pt2 = pt + stride;
    const bool two = pt2 < p.points;
    float gx[2], gy[2];
    {
      const float* xa = p.xin + ((long long)cloud * p.points + pt) * 3;
      const float* xb = p.xin + ((long long)cloud * p.points + (two ? pt2 : pt)) * 3;
      const float pa[3] = {__ldg(xa), __ldg(xa + 1), __ldg(xa + 2)}, pb[3] = {__ldg(xb), __ldg(xb + 1), __ldg(xb + 2)};
      lookup_coords(p, pa, c_in, fx, cx, fy, cy, gx[0], gy[0]);
      lookup_coords(p, pb, c_in, fx, cx, fy, cy, gx[1], gy[1]);
    }
    Taps taps[2][NCH];
#pragma unroll
    for (int h = 0; h < 2; ++h)
#pragma unroll
      for (int k = 0; k < NCH; ++k)
        if (ch_ptr[k] != nullptr) lookup_issue(ch_ptr[k], ch_h[k], ch_w[k], ch_c[k], gx[h], gy[h], taps[h][k]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      if (h == 1 && !two) break;
      const long long orow = (long long)cloud * p.rows_per_cloud + (h ? pt2 : pt);
#pragma unroll
      for (int k = 0; k < NCH; ++k) {
        if (ch_ptr[k] == nullptr) continue;
        float acc[8];
        lookup_blend(taps[h][k], acc);
        if (p.stats != nullptr) {
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const bool inA = j < bnd[k];
            sA1[k] += inA ? acc[j] : 0.f;
            sA2[k] += inA ? acc[j] * acc[j] : 0.f;
            sB1[k] += inA ? 0.f : acc[j];
            sB2[k] += inA ? 0.f : acc[j] * acc[j];
          }
        }
        if (p.out16 != nullptr) {
          *reinterpret_cast<uint4*>(p.out16 + orow * p.ldo16 + ch_col[k]) =
              make_uint4(pack_bf16x2(acc[0], acc[1]), pack_bf16x2(acc[2], acc[3]), pack_bf16x2(acc[4], acc[5]),
                         pack_bf16x2(acc[6], acc[7]));
        }
        if (p.out32 != nullptr) {
          float4* o = reinterpret_cast<float4*>(p.out32 + orow * p.ldo32 + ch_col[k]);
          o[0] = make_float4(acc[0], acc[1], acc[2], acc[3]);
          o[1] = make_float4(acc[4], acc[5], acc[6], acc[7]);
        }
      }
    }
  }
  if (p.stats != nullptr) {
#pragma unroll
    for (int k = 0; k < NCH; ++k) {
      if (ch_ptr[k] == nullptr) continue;
      atomicAdd(&sgrp[gA[k] * 2], static_cast<double>(sA1[k]));
      atomicAdd(&sgrp[gA[k] * 2 + 1], static_cast<double>(sA2[k]));
      if (bnd[k] < 8) {
        atomicAdd(&sgrp[(gA[k] + 1) * 2], static_cast<double>(sB1[k]));
        atomicAdd(&sgrp[(gA[k] + 1) * 2 + 1], static_cast<double>(sB2[k]));
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < p.stat_groups * 2; i += blockDim.x)
      atomicAdd(p.stats + (long long)cloud * p.stat_groups * 2 + i, sgrp[i]);
  }
}

// ---------------------------------------------------------------------------------------------
// Shared-memory staged lookup (the production path when the slice of one cloud's pyramid fits in shared memory).
//
// The legacy kernel above gathers 4 taps x sum(C) x 2 B = 5.4 KB per point from L2 (704 MB per launch at 64 clouds x 2048
// points), which bounds it at the L2 gather rate, far below the HBM roofline of its compulsory traffic (pyramid once +
// output once).  Here a CTA owns (cloud, channel slice, point range): slice s of S holds channels
// [s C_l / S, (s + 1) C_l / S) of every level, copied once into shared memory (cp.async, 16 B units, per-pixel runs stay
// contiguous), and all of the CTA's points gather from shared memory.  Per 256-point chunk one thread per point computes
// reparam -> projection -> tap geometry for every level into a small table (phase A); then thread (point lane, unit)
// blends UPT 8-channel units of one level for every point of its lane (phase B): the unit -> (level, column) mapping is
// fixed per thread, so the per-channel GroupNorm sums live in registers (packed fp32x2 arithmetic) and are reduced once
// per CTA.  Global traffic is the compulsory traffic: each pyramid byte is read once per point range, each output row
// segment is written once in runs of C_l / S channels.
constexpr int LS_THREADS = 512;
constexpr int LS_CHUNK = 256;                  // points per tap table
constexpr int LS_SGRP_BYTES = 64 * 2 * 8;      // per-group sums (stat_groups <= 64), double
constexpr size_t LS_SMEM_MAX = 227 * 1024;

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ uint64_t pack_f32x2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack_f32x2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t fma_f32x2(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ uint64_t add_f32x2(uint64_t a, uint64_t b) {
  uint64_t d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
// one bf16x2 word -> two fp32 lanes (exact)
__device__ __forceinline__ uint64_t bf16x2_to_f32x2(uint32_t v) {
  return pack_f32x2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u));
}

// Blend and statistics run on packed fp32x2 arithmetic (FFMA2 / FADD2).
// HYBRID: levels flagged in p.glob_mask are too large to stage (256^2 images: the 64 x 64 x 96 level is 786 KB per cloud);
// their threads gather the four taps from the L2-resident channels-last map instead, with the taps of the NEXT point in
// flight while the current one is blended, and the other levels still come from shared memory.  The large level is the
// one with the FEWEST channels, so the global gather shrinks from 4 x 672 to 4 x 96 channels per point.
template <int UPT, bool HYBRID = false>
__global__ void __launch_bounds__(LS_THREADS, 1) lookup_staged_kernel(const LookupP p, const int S, const int pts_per_cta) {
  extern __shared__ __align__(16) uint8_t lsm[];
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  const int slice = blockIdx.x, cloud = blockIdx.y, tid = threadIdx.x;
  const int pt_begin = blockIdx.z * pts_per_cta;
  const int pt_end = min(p.points, pt_begin + pts_per_cta);

  // geometry of this slice: 16 B units per pixel, byte offset of every level in shared memory, thread units per point
  int nU[GECCO_MAX_LEVELS], sm_off[GECCO_MAX_LEVELS], col_off[GECCO_MAX_LEVELS];
  int off = LS_SGRP_BYTES, tpp = 0, col = 0;  // [per-group sums][pyramid slice][tap tables]
#pragma unroll
  for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
    nU[l] = l < p.n_levels ? p.lvl_c[l] / (8 * S) : 0;
    sm_off[l] = off;
    col_off[l] = col;
    if (!(HYBRID && ((p.glob_mask >> l) & 1))) off += p.lvl_h[l] * p.lvl_w[l] * nU[l] * 16;
    tpp += nU[l] / UPT;
    col += p.lvl_c[l];
  }
  double* sgrp = reinterpret_cast<double*>(lsm);
  // two tap tables (chunk parity): [n_levels][LS_CHUNK] 4 x u16 pixel indices, then [n_levels][LS_CHUNK] 4 weights
  const int tab_bytes = p.n_levels * LS_CHUNK * 24;
  uint8_t* tab0 = lsm + off;

  // ---- stage the slice (asynchronously; the tap table of the first chunk is computed under it)
#pragma unroll
  for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
    if (nU[l] == 0) continue;
    if (HYBRID && ((p.glob_mask >> l) & 1)) continue;  // gathered from global memory
    const int C = p.lvl_c[l], n = nU[l];
    const int total = p.lvl_h[l] * p.lvl_w[l] * n;
    const __nv_bfloat16* src = p.lvl_ptr[l] + (long long)cloud * p.lvl_h[l] * p.lvl_w[l] * C + slice * n * 8;
    const uint32_t dst = smem_u32(lsm + sm_off[l]);
    for (int i = tid; i < total; i += LS_THREADS) {
      const int px = i / n, u = i - px * n;
      cp_async16(dst + i * 16, src + (long long)px * C + u * 8);
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");

  // ---- fixed (point lane, unit) role of this thread: units u0 + k nU / UPT of one level, so that consecutive threads
  // of a point read consecutive 16 B of a pixel (bank-conflict free) and write consecutive 16 B of the output row
  const int lanes = LS_THREADS / tpp;  // points in flight
  const int pl = tid / tpp, ut = tid - pl * tpp;
  const bool active = pl < lanes;
  int lv = 0, u0 = ut;
#pragma unroll
  for (int l = 0; l < GECCO_MAX_LEVELS - 1; ++l) {
    if (lv == l && u0 >= nU[l] / UPT) {
      u0 -= nU[l] / UPT;
      lv = l + 1;
    }
  }
  int my_n = 0, my_sm = 0, my_col = 0;
#pragma unroll
  for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
    if (l == lv) {
      my_n = nU[l];
      my_sm = sm_off[l];
      my_col = col_off[l] + slice * nU[l] * 8;
    }
  }
  const uint8_t* gbase = lsm + my_sm + u0 * 16;
  int gstride = my_n * 16;
  const int kstride = (my_n / UPT) * 16;  // bytes between the units of this thread
  bool my_glob = false;
  if constexpr (HYBRID) {
#pragma unroll
    for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
      if (l == lv && ((p.glob_mask >> l) & 1)) {
        my_glob = true;
        const int C = p.lvl_c[l];
        gbase = reinterpret_cast<const uint8_t*>(p.lvl_ptr[l] + (long long)cloud * p.lvl_h[l] * p.lvl_w[l] * C + slice * nU[l] * 8 + u0 * 8);
        gstride = C * 2;  // one pixel of the channels-last map
      }
    }
  }
  my_col += u0 * 8;
  const int kcol = (my_n / UPT) * 8;

  float s1[UPT][8], s2[UPT][8];
#pragma unroll
  for (int k = 0; k < UPT; ++k)
#pragma unroll
    for (int j = 0; j < 8; ++j) s1[k][j] = s2[k][j] = 0.f;

  float c_in = 1.f;
  if (p.sigma != nullptr) {
    const float sg = __ldg(p.sigma + (long long)cloud * p.sigma_stride);
    c_in = 1.0f / sqrtf(p.sigma_data * p.sigma_data + sg * sg);
  }
  const float* Kc = p.K + (long long)cloud * 9;
  const float fx = __ldg(Kc + 0), cx = __ldg(Kc + 2), fy = __ldg(Kc + 4), cy = __ldg(Kc + 5);

  // phase A: tap geometry of every level of one point (one thread per point of the chunk) into table `par`
  auto load_xyz = [&](int c0, float (&xyz)[3]) {
    const float* xp = p.xin + ((long long)cloud * p.points + min(c0 + tid, pt_end - 1)) * 3;
    xyz[0] = __ldg(xp); xyz[1] = __ldg(xp + 1); xyz[2] = __ldg(xp + 2);
  };
  auto write_taps = [&](int par, const float (&xyz)[3]) {
    float gx, gy;
    lookup_coords(p, xyz, c_in, fx, cx, fy, cy, gx, gy);
    uint2* tidx = reinterpret_cast<uint2*>(tab0 + par * tab_bytes);
    float4* tw = reinterpret_cast<float4*>(tab0 + par * tab_bytes + p.n_levels * LS_CHUNK * 8);
#pragma unroll
    for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
      if (l >= p.n_levels) break;
      int pix[4];
      float w[4];
      bool tv[4];
      lookup_geom(p.lvl_h[l], p.lvl_w[l], gx, gy, pix, w, tv);
      tidx[l * LS_CHUNK + tid] = make_uint2((uint32_t)pix[0] | ((uint32_t)pix[1] << 16), (uint32_t)pix[2] | ((uint32_t)pix[3] << 16));
      tw[l * LS_CHUNK + tid] = make_float4(w[0], w[1], w[2], w[3]);
    }
  };
  if (tid < LS_CHUNK && pt_begin < pt_end) {
    float xyz[3];
    load_xyz(pt_begin, xyz);
    write_taps(0, xyz);
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();

  int par = 0;
  for (int c0 = pt_begin; c0 < pt_end; c0 += LS_CHUNK, par ^= 1) {
    const int cn = min(LS_CHUNK, pt_end - c0);
    const bool prep_next = tid < LS_CHUNK && c0 + LS_CHUNK < pt_end;
    float xyz[3];
    if (prep_next) load_xyz(c0 + LS_CHUNK, xyz);  // in flight under phase B
    // ---- phase B: gather + blend from shared memory
    if (active) {
      const uint2* my_idx = reinterpret_cast<const uint2*>(tab0 + par * tab_bytes) + lv * LS_CHUNK;
      const float4* my_w = reinterpret_cast<const float4*>(tab0 + par * tab_bytes + p.n_levels * LS_CHUNK * 8) + lv * LS_CHUNK;
      // the table entry of the next point is fetched one iteration ahead (shortens the dependent LDS -> LDS chain)
      uint2 ix_n = make_uint2(0u, 0u);
      float4 w4_n = make_float4(0.f, 0.f, 0.f, 0.f);
      if (pl < cn) {
        ix_n = my_idx[pl];
        w4_n = my_w[pl];
      }
      [[maybe_unused]] uint4 qn[4][UPT];
      for (int i = pl; i < cn; i += lanes) {
        const uint2 ix = ix_n;
        const float4 w4 = w4_n;
        if (i + lanes < cn) {
          ix_n = my_idx[i + lanes];
          w4_n = my_w[i + lanes];
        }
        const uint32_t px[4] = {ix.x & 0xffffu, ix.x >> 16, ix.y & 0xffffu, ix.y >> 16};
        const float wt[4] = {w4.x, w4.y, w4.z, w4.w};
        uint4 q[4][UPT];
        if (HYBRID && my_glob) {
          // global (L2) gather, software pipelined: this point's taps were requested one iteration ago
          if (i == pl) {
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
              for (int k = 0; k < UPT; ++k) qn[t][k] = __ldg(reinterpret_cast<const uint4*>(gbase + (size_t)px[t] * gstride + k * kstride));
          }
#pragma unroll
          for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int k = 0; k < UPT; ++k) q[t][k] = qn[t][k];
          if (i + lanes < cn) {
            const uint32_t pn[4] = {ix_n.x & 0xffffu, ix_n.x >> 16, ix_n.y & 0xffffu, ix_n.y >> 16};
#pragma unroll
            for (int t = 0; t < 4; ++t)
#pragma unroll
              for (int k = 0; k < UPT; ++k) qn[t][k] = __ldg(reinterpret_cast<const uint4*>(gbase + (size_t)pn[t] * gstride + k * kstride));
          }
        } else {
#pragma unroll
          for (int t = 0; t < 4; ++t)
#pragma unroll
            for (int k = 0; k < UPT; ++k) q[t][k] = *reinterpret_cast<const uint4*>(gbase + px[t] * gstride + k * kstride);
        }
        __nv_bfloat16* orow = p.out16 + ((long long)cloud * p.rows_per_cloud + c0 + i) * p.ldo16 + my_col;
#pragma unroll
        for (int k = 0; k < UPT; ++k) {
          uint32_t o[4];
          uint64_t acc[4] = {0ull, 0ull, 0ull, 0ull};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const uint64_t ww = pack_f32x2(wt[t], wt[t]);
            acc[0] = fma_f32x2(bf16x2_to_f32x2(q[t][k].x), ww, acc[0]);
            acc[1] = fma_f32x2(bf16x2_to_f32x2(q[t][k].y), ww, acc[1]);
            acc[2] = fma_f32x2(bf16x2_to_f32x2(q[t][k].z), ww, acc[2]);
            acc[3] = fma_f32x2(bf16x2_to_f32x2(q[t][k].w), ww, acc[3]);
          }
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            uint64_t a1 = pack_f32x2(s1[k][2 * j], s1[k][2 * j + 1]), a2 = pack_f32x2(s2[k][2 * j], s2[k][2 * j + 1]);
            a1 = add_f32x2(a1, acc[j]);
            a2 = fma_f32x2(acc[j], acc[j], a2);
            unpack_f32x2(a1, s1[k][2 * j], s1[k][2 * j + 1]);
            unpack_f32x2(a2, s2[k][2 * j], s2[k][2 * j + 1]);
            float lo, hi;
            unpack_f32x2(acc[j], lo, hi);
            o[j] = pack_bf16x2(lo, hi);
          }
          *reinterpret_cast<uint4*>(orow + k * kcol) = make_uint4(o[0], o[1], o[2], o[3]);
        }
      }
    }
    if (prep_next) write_taps(par ^ 1, xyz);
    __syncthreads();
  }

  // ---- GroupNorm statistics (models/ray.py:53).  Deterministic: every thread parks its per-column sums in shared memory
  // (the pyramid slice is no longer needed), one thread per column adds the point lanes in a fixed order, and only the
  // per-group / global accumulation uses (double) atomics.
  if (p.stats != nullptr) {
    float* red = reinterpret_cast<float*>(lsm + LS_SGRP_BYTES);  // [2][lanes][ctot]
    for (int i = tid; i < p.stat_groups * 2; i += LS_THREADS) sgrp[i] = 0.0;
    if (active) {
#pragma unroll
      for (int k = 0; k < UPT; ++k)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          red[pl * p.ctot + my_col + k * kcol + j] = s1[k][j];
          red[(lanes + pl) * p.ctot + my_col + k * kcol + j] = s2[k][j];
        }
    }
    __syncthreads();
    const int gsz = p.ctot / p.stat_groups;
    for (int i = tid; i < p.ctot; i += LS_THREADS) {
      // column i belongs to this slice if it lies in [slice C_l / S, (slice + 1) C_l / S) of its level
      bool mine = false;
#pragma unroll
      for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
        const int c = i - col_off[l];
        if (nU[l] > 0 && c >= 0 && c < p.lvl_c[l]) mine = c / (nU[l] * 8) == slice;
      }
      if (!mine) continue;
      double a = 0.0, b = 0.0;
      for (int q = 0; q < lanes; ++q) {
        a += static_cast<double>(red[q * p.ctot + i]);
        b += static_cast<double>(red[(lanes + q) * p.ctot + i]);
      }
      atomicAdd(&sgrp[(i / gsz) * 2], a);
      atomicAdd(&sgrp[(i / gsz) * 2 + 1], b);
    }
    __syncthreads();
    for (int i = tid; i < p.stat_groups * 2; i += LS_THREADS)
      if (sgrp[i] != 0.0) atomicAdd(p.stats + (long long)cloud * p.stat_groups * 2 + i, sgrp[i]);
  }
}

// Slice count of the staged kernel: the smallest S that divides every level into whole 8-channel units, fits one
// slice of one cloud (plus the tap table) in shared memory and gives every unit a thread.  0 = not applicable.
// GECCO_LOOKUP_SLICES overrides (0 forces the legacy global-gather kernel).
struct StagedPlan {
  int S, upt;
  size_t smem;
  int glob_mask;  // levels left in global memory (hybrid kernel)
};
StagedPlan plan_staged(const LookupP& p, int stat_groups) {
  StagedPlan none = {0, 0, 0, 0};
  if (p.out16 == nullptr || p.out32 != nullptr) return none;
  if (stat_groups > 64) return none;
  int forced = -1;
  if (const char* v = getenv("GECCO_LOOKUP_SLICES")) forced = atoi(v);
  if (forced == 0) return none;
  for (int l = 0; l < p.n_levels; ++l)
    if (p.lvl_h[l] * p.lvl_w[l] > 65535) return none;
  // Measured at 64 clouds x 2048 points (tools/lookup_time.py): 137^2 pyramids (S = 2) 105 us against 228 us for the
  // global-gather kernel; 256^2 pyramids need S = 12 (7 threads per point, a tap-table entry per 8 channels) and are
  // slower than the global gather (270 against 236 us), so the automatic choice stops at S = 4.
  // Hybrid plans: first everything staged; if no S <= 4 fits, the level with the largest map (the fewest channels in a
  // CNN pyramid) stays in global memory and only the others are staged.
  const bool hybrid_ok = p.n_levels >= 2;
  int biggest = 0;
  for (int l = 1; l < p.n_levels; ++l)
    if ((size_t)p.lvl_h[l] * p.lvl_w[l] * p.lvl_c[l] > (size_t)p.lvl_h[biggest] * p.lvl_w[biggest] * p.lvl_c[biggest]) biggest = l;
  static const int cand[] = {1, 2, 3, 4, 6, 8, 12, 16, 24, 32, 48};
  for (int pass = 0; pass < (hybrid_ok && forced < 0 ? 2 : 1); ++pass)
  for (int S : cand) {
    const int glob_mask = pass == 1 ? (1 << biggest) : 0;
    if (forced > 0 && S != forced) continue;
    if (forced < 0 && S > 4) break;
    bool ok = true, even = true;
    size_t bytes = 0;
    int units = 0;
    for (int l = 0; l < p.n_levels; ++l) {
      if (p.lvl_c[l] % (8 * S) != 0) { ok = false; break; }
      const int n = p.lvl_c[l] / (8 * S);
      even = even && (n % 2 == 0);
      units += n;
      if (!((glob_mask >> l) & 1)) bytes += (size_t)p.lvl_h[l] * p.lvl_w[l] * n * 16;
    }
    if (!ok) continue;
    const int upt = even ? 2 : 1;
    if (units / upt > LS_THREADS) continue;
    const size_t tab = (size_t)2 * p.n_levels * LS_CHUNK * 24;  // two tap tables
    // the statistics epilogue reuses the slice + tables for [2][point lanes][ctot] floats
    const size_t red = (size_t)2 * (LS_THREADS / (units / upt)) * p.ctot * 4;
    size_t total = bytes + tab;
    if (red > total) total = red;
    total += LS_SGRP_BYTES;
    if (total > LS_SMEM_MAX) continue;
    return {S, upt, total, glob_mask};
  }
  return none;
}

// GroupNorm (no affine) followed by Linear, folded per cloud (models/ray.py:52-55):
//   Linear(GN(z))[o] = sum_c (W[o,c] rstd_g(c)) z[c] + (b[o] - sum_c W[o,c] mean_g(c) rstd_g(c))
constexpr int FGN_ROWS = 16;  // output rows per block (4 warps x 4)

__global__ void __launch_bounds__(128)
fold_gn_kernel(const float* __restrict__ W, const float* __restrict__ bias, const double* __restrict__ stats, double count,
               float eps, int groups, int c_in, int c_out, __nv_bfloat16* __restrict__ wb, long long ldwb,
               float* __restrict__ bb) {
  __shared__ float smean[64], srstd[64];
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  const int cloud = blockIdx.y;
  const int gs = c_in / groups;
  const double* cs = stats + (long long)cloud * groups * 2;
  for (int g = threadIdx.x; g < groups; g += blockDim.x) {  // the only double precision arithmetic
    const double m = cs[g * 2] / count;
    double var = cs[g * 2 + 1] / count - m * m;
    if (var < 0.0) var = 0.0;
    smean[g] = static_cast<float>(m);
    srstd[g] = static_cast<float>(1.0 / sqrt(var + (double)eps));
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int o_end = min((int)(blockIdx.x + 1) * FGN_ROWS, c_out);
  for (int o = blockIdx.x * FGN_ROWS + warp; o < o_end; o += 4) {
    const float* wr = W + (long long)o * c_in;
    __nv_bfloat16* dst = wb + ((long long)cloud * c_out + o) * ldwb;
    float acc = 0.f;
#pragma unroll 4
    for (int c = lane * 2; c < c_in; c += 64) {
      const float2 w2 = __ldg(reinterpret_cast<const float2*>(wr + c));
      const int g0 = c / gs, g1 = (c + 1) / gs;
      const float w0 = w2.x * srstd[g0], w1 = w2.y * srstd[g1];
      *reinterpret_cast<uint32_t*>(dst + c) = pack_bf16x2(w0, w1);
      acc += w0 * smean[g0] + w1 * smean[g1];
    }
    acc = warp_sum(acc);
    if (lane == 0) bb[(long long)cloud * c_out + o] = __ldg(bias + o) - acc;
  }
}

// fp32 NCHW -> bf16 NHWC (per image), via a 32x32 smem transpose tile over (C, H*W).
__global__ void nchw_to_nhwc_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int C, int HW) {
  __shared__ float tile[32][33];
  const int img = blockIdx.z;
  const int c0 = blockIdx.y * 32, p0 = blockIdx.x * 32;
  const float* s = src + (long long)img * C * HW;
  __nv_bfloat16* d = dst + (long long)img * C * HW;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i, pix = p0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && pix < HW) ? s[(long long)c * HW + pix] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int pix = p0 + i, c = c0 + threadIdx.x;
    if (c < C && pix < HW) d[(long long)pix * C + c] = __float2bfloat16(tile[threadIdx.x][i]);
  }
}

}  // namespace

int launch_lookup(const gecco_lookup_args& a, cudaStream_t s) {
  GECCO_REQUIRE(a.n_levels >= 1 && a.n_levels <= GECCO_MAX_LEVELS, "lookup: 1..%d pyramid levels supported", GECCO_MAX_LEVELS);
  GECCO_REQUIRE(a.reparam >= 0 && a.reparam <= 2, "lookup: unknown reparam %d", a.reparam);
  GECCO_REQUIRE(a.xin && a.K, "lookup: xin and K are required");
  GECCO_REQUIRE(a.out_bf16 || a.out_f32, "lookup: no output");
  LookupP p;
  p.xin = a.xin; p.sigma = a.sigma; p.sigma_stride = a.sigma_stride; p.sigma_data = a.sigma_data;
  p.reparam = a.reparam;
  for (int j = 0; j < 3; ++j) { p.mean[j] = a.mean[j]; p.rsig[j] = a.sigma_r[j]; }
  p.logit_scale = a.logit_scale;
  p.K = a.K;
  p.n_levels = a.n_levels;
  int ctot = 0;
  for (int l = 0; l < GECCO_MAX_LEVELS; ++l) {
    p.lvl_ptr[l] = nullptr; p.lvl_h[l] = p.lvl_w[l] = p.lvl_c[l] = 0;
  }
  for (int l = 0; l < a.n_levels; ++l) {
    GECCO_REQUIRE(a.level_ptr[l] && a.level_c[l] % 8 == 0 && a.level_h[l] > 0 && a.level_w[l] > 0,
                  "lookup: level %d must be non-empty with a channel count that is a multiple of 8", l);
    p.lvl_ptr[l] = static_cast<const __nv_bfloat16*>(a.level_ptr[l]);
    p.lvl_h[l] = a.level_h[l]; p.lvl_w[l] = a.level_w[l]; p.lvl_c[l] = a.level_c[l];
    ctot += a.level_c[l];
  }
  GECCO_REQUIRE(ctot <= 32 * 8 * LK_MAXCH, "lookup: at most %d channels supported", 32 * 8 * LK_MAXCH);
  GECCO_REQUIRE(!a.out_bf16 || a.ldo16 % 8 == 0, "lookup: bf16 leading dimension must be a multiple of 8");
  GECCO_REQUIRE(!a.out_f32 || a.ldo32 % 4 == 0, "lookup: fp32 leading dimension must be a multiple of 4");
  GECCO_REQUIRE(!a.stats || (a.stat_groups > 0 && ctot % a.stat_groups == 0), "lookup: bad statistics groups");
  p.points = a.points; p.rows_per_cloud = a.rows_per_cloud; p.ctot = ctot;
  p.out16 = static_cast<__nv_bfloat16*>(a.out_bf16); p.ldo16 = a.ldo16;
  p.out32 = a.out_f32; p.ldo32 = a.ldo32;
  p.stats = a.stats; p.stat_groups = a.stats ? a.stat_groups : 0;
  if (a.points == 0 || a.clouds == 0) return GECCO_OK;
  GECCO_REQUIRE(!a.stats || ctot / a.stat_groups >= 8, "lookup: GroupNorm groups must be at least 8 channels wide");
  p.glob_mask = 0;
  const StagedPlan plan = plan_staged(p, p.stat_groups);
  if (plan.S > 0) {
    p.glob_mask = plan.glob_mask;
    // (slice, cloud, point range): point ranges only when clouds x slices leave SMs idle
    int z = sm_count() / (a.clouds * plan.S);
    if (z < 1) z = 1;
    int per = ceil_div(ceil_div(a.points, z), 32) * 32;
    z = ceil_div(a.points, per);
    dim3 grid(plan.S, a.clouds, z);
    auto go = [&](auto kern, bool& done) {
      if (!done) {
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)LS_SMEM_MAX);
        done = true;
      }
      launch_small(kern, grid, dim3(LS_THREADS), plan.smem, s, p, plan.S, per);
    };
    static bool attr_done[4] = {false, false, false, false};
    if (plan.glob_mask != 0 && plan.upt == 2) go(lookup_staged_kernel<2, true>, attr_done[2]);
    else if (plan.glob_mask != 0) go(lookup_staged_kernel<1, true>, attr_done[3]);
    else if (plan.upt == 2) go(lookup_staged_kernel<2>, attr_done[0]);
    else go(lookup_staged_kernel<1>, attr_done[1]);
    GECCO_CHECK_LAUNCH("lookup_staged_kernel");
    return GECCO_OK;
  }
  dim3 grid(ceil_div(a.points, LK_WARPS * LK_POINTS_PER_WARP), a.clouds);
  const size_t sm = p.stat_groups * 2 * sizeof(double);
  switch (ceil_div(ctot, 256)) {
    case 1: lookup_kernel<1><<<grid, LK_WARPS * 32, sm, s>>>(p); break;
    case 2: lookup_kernel<2><<<grid, LK_WARPS * 32, sm, s>>>(p); break;
    case 3: lookup_kernel<3><<<grid, LK_WARPS * 32, sm, s>>>(p); break;
    default: lookup_kernel<4><<<grid, LK_WARPS * 32, sm, s>>>(p); break;
  }
  GECCO_CHECK_LAUNCH("lookup_kernel");
  return GECCO_OK;
}

int launch_fold_gn(const float* W, const float* bias, const double* stats, double count, float eps, int groups,
                   int c_in, int c_out, int clouds, void* wb, long long ldwb, float* bb, cudaStream_t s) {
  GECCO_REQUIRE(groups > 0 && groups <= 64 && c_in % groups == 0 && c_in % 2 == 0 && ldwb % 2 == 0, "fold_gn: bad layout");
  dim3 grid(ceil_div(c_out, FGN_ROWS), clouds);
  launch_small(fold_gn_kernel, grid, dim3(128), 0, s, W, bias, stats, count, eps, groups, c_in, c_out, static_cast<__nv_bfloat16*>(wb),
               ldwb, bb);
  GECCO_CHECK_LAUNCH("fold_gn_kernel");
  return GECCO_OK;
}

}  // namespace gecco

extern "C" int gecco_lookup(const gecco_lookup_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_lookup: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_lookup(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_fold_group_norm(const float* w, const float* bias, const double* stats, double count, float eps,
                                     int32_t groups, int32_t c_in, int32_t c_out, int32_t clouds, void* w_folded_bf16,
                                     int64_t ldw, float* bias_folded, void* stream) {
  return gecco::launch_fold_gn(w, bias, stats, count, eps, groups, c_in, c_out, clouds, w_folded_bf16, ldw, bias_folded,
                               static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_pack_features(const float* nchw, void* nhwc_bf16, int32_t images, int32_t c, int32_t h, int32_t w,
                                   void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(nchw && nhwc_bf16 && images > 0 && c > 0 && h > 0 && w > 0, "pack_features: bad arguments");
  dim3 grid(ceil_div(h * w, 32), ceil_div(c, 32), images);
  nchw_to_nhwc_bf16_kernel<<<grid, dim3(32, 8), 0, static_cast<cudaStream_t>(stream)>>>(
      nchw, static_cast<__nv_bfloat16*>(nhwc_bf16), c, h * w);
  GECCO_CHECK_LAUNCH("nchw_to_nhwc_bf16_kernel");
  return GECCO_OK;
}
