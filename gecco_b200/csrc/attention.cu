// Inducer-point attention (models/set_transformer.py):
//   pool   (AttentionPool.forward :47-65): 64 learned queries attend over the N points of a cloud;
//          split over key ranges (flash-decoding regime) + a small combine kernel.
//   unpool (nn.MultiheadAttention :90,112): every point attends over the 64 inducers.
// Warp-level mma.sync (m16n8k16 bf16, fp32 accumulate) kernels with cp.async staging; K/V/Q come from the bf16
// projections written by the tcgen05 GEMM.  The unpool core also exists on tcgen05 / TMEM (attention_tc.cu), which
// launch_unpool_attention prefers where its shape constraints hold; likewise the pool core (attention_pool_tc.cu).
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

#include <stdlib.h>

namespace gecco {

namespace {

constexpr int NI = 64;       // inducers (queries of pool / keys of unpool)
constexpr int KT = 64;       // key tile of the pool kernel
constexpr int PAD = 8;       // bf16 padding per smem row (keeps ldmatrix conflict-free)

__device__ __forceinline__ void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(smem_u32(p)));
}
__device__ __forceinline__ void mma16816(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
// ex2.approx: one MUFU instruction (exp2f adds range handling that softmax on max-subtracted scores does not need;
// ex2.approx(-inf) = +0)
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// ------------------------------------------------------------------------------------------------
// pool: grid (splits, heads, clouds), 128 threads; warp w owns inducers 16w..16w+15.
// q_ind: bf16 [heads][64][D], pre-multiplied by softmax_scale * log2(e).
// part : fp32 [clouds][heads][splits][64][D + 2]  (unnormalised O, running max (log2 domain), sum)
template <int D>
__global__ void __launch_bounds__(128)
pool_attn_kernel(const __nv_bfloat16* __restrict__ kv, long long ld, int k_off, int v_off, int rows_per_cloud,
                 int valid_rows, const __nv_bfloat16* __restrict__ q_ind, float* __restrict__ part, int tiles_per_split) {
  constexpr int LDS = D + PAD;
  constexpr int CH = D / 8;  // 16-byte chunks per row
  constexpr int PS = 3;  // cp.async stages: two key tiles in flight while one is consumed, one barrier per tile
  extern __shared__ __align__(16) uint8_t pool_smem[];
  __nv_bfloat16(*sQ)[LDS] = reinterpret_cast<__nv_bfloat16(*)[LDS]>(pool_smem);
  __nv_bfloat16(*sK)[KT][LDS] = reinterpret_cast<__nv_bfloat16(*)[KT][LDS]>(pool_smem + NI * LDS * 2);
  __nv_bfloat16(*sV)[KT][LDS] = reinterpret_cast<__nv_bfloat16(*)[KT][LDS]>(pool_smem + (NI + PS * KT) * LDS * 2);

  const int split = blockIdx.x, head = blockIdx.y, cloud = blockIdx.z;
  const int nsplit = gridDim.x, heads = gridDim.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;

  const int n_tiles = (valid_rows + KT - 1) / KT;
  const int tile0 = split * tiles_per_split;
  const int tile1 = min(tile0 + tiles_per_split, n_tiles);

  const __nv_bfloat16* kbase = kv + ((long long)cloud * rows_per_cloud) * ld + k_off + head * D;
  const __nv_bfloat16* vbase = kv + ((long long)cloud * rows_per_cloud) * ld + v_off + head * D;

  auto stage = [&](int buf, int tile) {
    const int key0 = tile * KT;
    for (int i = threadIdx.x; i < KT * CH; i += 128) {
      const int r = i / CH, c = i % CH;
      cp_async16(&sK[buf][r][c * 8], kbase + (long long)(key0 + r) * ld + c * 8);
      cp_async16(&sV[buf][r][c * 8], vbase + (long long)(key0 + r) * ld + c * 8);
    }
  };

  // queries -> smem -> A fragments
  for (int i = threadIdx.x; i < NI * CH; i += 128) {
    const int r = i / CH, c = i % CH;
    *reinterpret_cast<uint4*>(&sQ[r][c * 8]) =
        __ldg(reinterpret_cast<const uint4*>(q_ind + ((long long)head * NI + r) * D + c * 8));
  }
  if (tile0 < tile1) stage(0, tile0);
  cp_async_commit();
  if (tile0 + 1 < tile1) stage(1, tile0 + 1);
  cp_async_commit();
  __syncthreads();
  uint32_t aQ[D / 16][4];
#pragma unroll
  for (int ks = 0; ks < D / 16; ++ks) ldsm_x4(aQ[ks], &sQ[16 * warp + (lane & 15)][ks * 16 + (lane >> 4) * 8]);

  float oacc[D / 8][4];
#pragma unroll
  for (int i = 0; i < D / 8; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) oacc[i][j] = 0.f;
  float m_run[2] = {-INFINITY, -INFINITY}, l_run[2] = {0.f, 0.f};

  for (int tile = tile0; tile < tile1; ++tile) {
    const int buf = (tile - tile0) % PS;
    cp_async_wait<1>();  // tile `tile` has landed (at most the group of tile + 1 is still in flight)
    __syncthreads();     // ... for every thread, and everybody is done with the buffer tile + 2 is about to overwrite
    if (tile + 2 < tile1) stage((buf + 2) % PS, tile + 2);
    cp_async_commit();

    // S = Q K^T  (16 x 64 per warp)
    float sacc[KT / 8][4];
#pragma unroll
    for (int i = 0; i < KT / 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sacc[i][j] = 0.f;
#pragma unroll
    for (int nb = 0; nb < KT / 8; nb += 2) {
#pragma unroll
      for (int ks = 0; ks < D / 16; ++ks) {
        uint32_t b[4];
        const int mid = lane >> 3, row = lane & 7;
        ldsm_x4(b, &sK[buf][8 * nb + (mid >> 1) * 8 + row][ks * 16 + (mid & 1) * 8]);
        mma16816(sacc[nb], aQ[ks], b[0], b[1]);
        mma16816(sacc[nb + 1], aQ[ks], b[2], b[3]);
      }
    }
    // mask padding keys, online softmax (base-2 domain)
    const int key0 = tile * KT;
    float tmax[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nb = 0; nb < KT / 8; ++nb) {
      const int kk = key0 + nb * 8 + 2 * t;
      if (kk >= valid_rows) { sacc[nb][0] = -INFINITY; sacc[nb][2] = -INFINITY; }
      if (kk + 1 >= valid_rows) { sacc[nb][1] = -INFINITY; sacc[nb][3] = -INFINITY; }
      tmax[0] = fmaxf(tmax[0], fmaxf(sacc[nb][0], sacc[nb][1]));
      tmax[1] = fmaxf(tmax[1], fmaxf(sacc[nb][2], sacc[nb][3]));
    }
    float alpha[2], muse[2];
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const float mnew = fmaxf(m_run[r], quad_max(tmax[r]));
      muse[r] = (mnew == -INFINITY) ? 0.f : mnew;
      alpha[r] = fast_exp2(m_run[r] - muse[r]);
      m_run[r] = mnew;
      l_run[r] *= alpha[r];
    }
#pragma unroll
    for (int i = 0; i < D / 8; ++i) {
      oacc[i][0] *= alpha[0]; oacc[i][1] *= alpha[0];
      oacc[i][2] *= alpha[1]; oacc[i][3] *= alpha[1];
    }
    uint32_t aP[KT / 16][4];
#pragma unroll
    for (int nb = 0; nb < KT / 8; ++nb) {
      const float p0 = fast_exp2(sacc[nb][0] - muse[0]), p1 = fast_exp2(sacc[nb][1] - muse[0]);
      const float p2 = fast_exp2(sacc[nb][2] - muse[1]), p3 = fast_exp2(sacc[nb][3] - muse[1]);
      l_run[0] += p0 + p1;
      l_run[1] += p2 + p3;
      aP[nb >> 1][(nb & 1) * 2 + 0] = pack_bf16x2(p0, p1);
      aP[nb >> 1][(nb & 1) * 2 + 1] = pack_bf16x2(p2, p3);
    }
    // O += P V
#pragma unroll
    for (int ks = 0; ks < KT / 16; ++ks) {
#pragma unroll
      for (int nb = 0; nb < D / 8; nb += 2) {
        uint32_t b[4];
        const int mid = lane >> 3, row = lane & 7;
        ldsm_x4_t(b, &sV[buf][16 * ks + (mid & 1) * 8 + row][8 * nb + (mid >> 1) * 8]);
        mma16816(oacc[nb], aP[ks], b[0], b[1]);
        mma16816(oacc[nb + 1], aP[ks], b[2], b[3]);
      }
    }
  }
  cp_async_wait<0>();

  l_run[0] = quad_sum(l_run[0]);
  l_run[1] = quad_sum(l_run[1]);
  float* prow = part + ((((long long)cloud * heads + head) * nsplit + split) * NI) * (D + 2);
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    float* pr = prow + (long long)(16 * warp + g + 8 * r) * (D + 2);
#pragma unroll
    for (int nb = 0; nb < D / 8; ++nb)
      *reinterpret_cast<float2*>(pr + nb * 8 + 2 * t) = make_float2(oacc[nb][2 * r], oacc[nb][2 * r + 1]);
    if (t == 0) {
      pr[D] = m_run[r];
      pr[D + 1] = l_run[r];
    }
  }
}

// combine the key-range partials: one warp per (cloud, head, inducer); "b h i d -> b i (h d)".
__global__ void pool_combine_kernel(const float* __restrict__ part, int heads, int nsplit, int D,
                                    __nv_bfloat16* __restrict__ out, long long ldo, int total_rows) {
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (wid >= total_rows) return;
  const int i = wid % NI;
  const int head = (wid / NI) % heads;
  const int cloud = wid / (NI * heads);
  const float* base = part + (((long long)cloud * heads + head) * nsplit) * NI * (D + 2);
  float M = -INFINITY;
  for (int s = 0; s < nsplit; ++s) M = fmaxf(M, base[((long long)s * NI + i) * (D + 2) + D]);
  float L = 0.f;
  float acc[2] = {0.f, 0.f};
  for (int s = 0; s < nsplit; ++s) {
    const float* pr = base + ((long long)s * NI + i) * (D + 2);
    const float m = pr[D];
    const float w = (m == -INFINITY) ? 0.f : fast_exp2(m - M);
    L += w * pr[D + 1];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int d = lane + 32 * j;
      if (d < D) acc[j] += w * pr[d];
    }
  }
  const float inv = 1.0f / L;
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int d = lane + 32 * j;
    if (d < D) out[((long long)cloud * NI + i) * ldo + head * D + d] = __float2bfloat16(acc[j] * inv);
  }
}

// ------------------------------------------------------------------------------------------------
// unpool: grid (row tiles of 128, clouds), 256 threads; warp w owns rows 16w..16w+15 of the tile and
// loops over heads.  q (pre-scaled by softmax_scale*log2e through the projection weights), k, v are bf16.
template <int D>
__global__ void __launch_bounds__(256)
unpool_attn_kernel(const __nv_bfloat16* __restrict__ q, long long ldq, const __nv_bfloat16* __restrict__ khv,
                   long long ldkv, int v_off, int rows_per_cloud, int heads, __nv_bfloat16* __restrict__ out,
                   long long ldo) {
  constexpr int LDS = D + PAD;
  constexpr int CH = D / 8;
  constexpr int RT = 128;
  extern __shared__ __align__(16) uint8_t smem_dyn[];
  // per stage: Q [128][LDS], K [64][LDS], V [64][LDS]
  constexpr int STAGE_ELEMS = (RT + 2 * NI) * LDS;
  __nv_bfloat16* sbase = reinterpret_cast<__nv_bfloat16*>(smem_dyn);

  const int cloud = blockIdx.y;
  const int row0 = blockIdx.x * RT;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane >> 2, t = lane & 3;

  const __nv_bfloat16* qbase = q + ((long long)cloud * rows_per_cloud + row0) * ldq;
  const __nv_bfloat16* kbase = khv + ((long long)cloud * NI) * ldkv;
  __nv_bfloat16* obase = out + ((long long)cloud * rows_per_cloud + row0) * ldo;

  auto stage = [&](int buf, int head) {
    __nv_bfloat16* sQ = sbase + buf * STAGE_ELEMS;
    __nv_bfloat16* sK = sQ + RT * LDS;
    __nv_bfloat16* sV = sK + NI * LDS;
    for (int i = threadIdx.x; i < RT * CH; i += 256) {
      const int r = i / CH, c = i % CH;
      cp_async16(sQ + r * LDS + c * 8, qbase + (long long)r * ldq + head * D + c * 8);
    }
    for (int i = threadIdx.x; i < NI * CH; i += 256) {
      const int r = i / CH, c = i % CH;
      cp_async16(sK + r * LDS + c * 8, kbase + (long long)r * ldkv + head * D + c * 8);
      cp_async16(sV + r * LDS + c * 8, kbase + (long long)r * ldkv + v_off + head * D + c * 8);
    }
  };

  stage(0, 0);
  cp_async_commit();
  for (int head = 0; head < heads; ++head) {
    const int buf = head & 1;
    if (head + 1 < heads) stage(buf ^ 1, head + 1);
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();
    __nv_bfloat16* sQ = sbase + buf * STAGE_ELEMS;
    __nv_bfloat16* sK = sQ + RT * LDS;
    __nv_bfloat16* sV = sK + NI * LDS;

    uint32_t aQ[D / 16][4];
#pragma unroll
    for (int ks = 0; ks < D / 16; ++ks) ldsm_x4(aQ[ks], sQ + (16 * warp + (lane & 15)) * LDS + ks * 16 + (lane >> 4) * 8);
    float sacc[NI / 8][4];
#pragma unroll
    for (int i = 0; i < NI / 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) sacc[i][j] = 0.f;
#pragma unroll
    for (int nb = 0; nb < NI / 8; nb += 2) {
#pragma unroll
      for (int ks = 0; ks < D / 16; ++ks) {
        uint32_t b[4];
        const int mid = lane >> 3, row = lane & 7;
        ldsm_x4(b, sK + (8 * nb + (mid >> 1) * 8 + row) * LDS + ks * 16 + (mid & 1) * 8);
        mma16816(sacc[nb], aQ[ks], b[0], b[1]);
        mma16816(sacc[nb + 1], aQ[ks], b[2], b[3]);
      }
    }
    float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
    for (int nb = 0; nb < NI / 8; ++nb) {
      mx[0] = fmaxf(mx[0], fmaxf(sacc[nb][0], sacc[nb][1]));
      mx[1] = fmaxf(mx[1], fmaxf(sacc[nb][2], sacc[nb][3]));
    }
    mx[0] = quad_max(mx[0]);
    mx[1] = quad_max(mx[1]);
    float sum[2] = {0.f, 0.f};
    uint32_t aP[NI / 16][4];
#pragma unroll
    for (int nb = 0; nb < NI / 8; ++nb) {
      const float p0 = fast_exp2(sacc[nb][0] - mx[0]), p1 = fast_exp2(sacc[nb][1] - mx[0]);
      const float p2 = fast_exp2(sacc[nb][2] - mx[1]), p3 = fast_exp2(sacc[nb][3] - mx[1]);
      sum[0] += p0 + p1;
      sum[1] += p2 + p3;
      aP[nb >> 1][(nb & 1) * 2 + 0] = pack_bf16x2(p0, p1);
      aP[nb >> 1][(nb & 1) * 2 + 1] = pack_bf16x2(p2, p3);
    }
    sum[0] = quad_sum(sum[0]);
    sum[1] = quad_sum(sum[1]);
    float oacc[D / 8][4];
#pragma unroll
    for (int i = 0; i < D / 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) oacc[i][j] = 0.f;
#pragma unroll
    for (int ks = 0; ks < NI / 16; ++ks) {
#pragma unroll
      for (int nb = 0; nb < D / 8; nb += 2) {
        uint32_t b[4];
        const int mid = lane >> 3, row = lane & 7;
        ldsm_x4_t(b, sV + (16 * ks + (mid & 1) * 8 + row) * LDS + 8 * nb + (mid >> 1) * 8);
        mma16816(oacc[nb], aP[ks], b[0], b[1]);
        mma16816(oacc[nb + 1], aP[ks], b[2], b[3]);
      }
    }
    // normalise, park the 16 x D result in this warp's (now consumed) Q rows, then store 16 B chunks
    const float inv0 = 1.0f / sum[0], inv1 = 1.0f / sum[1];
    __syncwarp();
#pragma unroll
    for (int nb = 0; nb < D / 8; ++nb) {
      *reinterpret_cast<uint32_t*>(sQ + (16 * warp + g) * LDS + nb * 8 + 2 * t) =
          pack_bf16x2(oacc[nb][0] * inv0, oacc[nb][1] * inv0);
      *reinterpret_cast<uint32_t*>(sQ + (16 * warp + g + 8) * LDS + nb * 8 + 2 * t) =
          pack_bf16x2(oacc[nb][2] * inv1, oacc[nb][3] * inv1);
    }
    __syncwarp();
    for (int i = lane; i < 16 * CH; i += 32) {
      const int r = 16 * warp + i / CH, c = i % CH;
      *reinterpret_cast<uint4*>(obase + (long long)r * ldo + head * D + c * 8) =
          *reinterpret_cast<const uint4*>(sQ + r * LDS + c * 8);
    }
    __syncthreads();
  }
  cp_async_wait<0>();
}

}  // namespace

// GECCO_POOL_TC=0 keeps the mma.sync kernel even where the tcgen05 kernel applies (A/B measurements).
static bool pool_tc_enabled() {
  const char* v = getenv("GECCO_POOL_TC");
  return !(v != nullptr && v[0] == '0');
}

int launch_pool_attention_partial(const gecco_pool_args& a, cudaStream_t s, int* splits_used) {
  *splits_used = 1;
  if (pool_tc_enabled() && pool_tc_supported(a)) return launch_pool_tc(a, s, splits_used);
  return launch_pool_attention(a, s);
}

int launch_pool_attention(const gecco_pool_args& a, cudaStream_t s) {
  if (pool_tc_enabled() && pool_tc_supported(a)) {
    int nsplit = 1;
    if (int rc = launch_pool_tc(a, s, &nsplit)) return rc;
    if (nsplit > 1) {
      const int rows = a.clouds * a.heads * NI;
      pool_combine_kernel<<<ceil_div(rows, 4), 128, 0, s>>>(a.partial, a.heads, nsplit, a.head_dim,
                                                           static_cast<__nv_bfloat16*>(a.out_bf16), a.ldo, rows);
      GECCO_CHECK_LAUNCH("pool_combine_kernel");
    }
    return GECCO_OK;
  }
  GECCO_REQUIRE(a.inducers == NI, "pool attention: only 64 inducers are supported (got %d)", a.inducers);
  GECCO_REQUIRE(a.head_dim == 32 || a.head_dim == 48 || a.head_dim == 64, "pool attention: head_dim must be 32, 48 or 64 (got %d)", a.head_dim);
  GECCO_REQUIRE(a.rows_per_cloud % KT == 0, "pool attention: rows_per_cloud must be a multiple of 64");
  GECCO_REQUIRE(a.ld % 8 == 0 && a.k_off % 8 == 0 && a.v_off % 8 == 0 && a.ldo % 2 == 0, "pool attention: misaligned layout");
  GECCO_REQUIRE(a.splits >= 1, "pool attention: splits must be >= 1");
  const int n_tiles = ceil_div(a.valid_rows, KT);
  const int tps = ceil_div(n_tiles, a.splits);
  dim3 grid(a.splits, a.heads, a.clouds);
  const __nv_bfloat16* kv = static_cast<const __nv_bfloat16*>(a.kv);
  const __nv_bfloat16* qi = static_cast<const __nv_bfloat16*>(a.q_inducers);
  const int smem = (NI + 2 * 3 * KT) * (a.head_dim + PAD) * 2;  // sQ + 3 stages of K and V
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(pool_attn_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pool_attn_kernel<48>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(pool_attn_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(pool_attn_kernel)");
    attr_set = true;
  }
  switch (a.head_dim) {
    case 32: pool_attn_kernel<32><<<grid, 128, smem, s>>>(kv, a.ld, a.k_off, a.v_off, a.rows_per_cloud, a.valid_rows, qi, a.partial, tps); break;
    case 48: pool_attn_kernel<48><<<grid, 128, smem, s>>>(kv, a.ld, a.k_off, a.v_off, a.rows_per_cloud, a.valid_rows, qi, a.partial, tps); break;
    default: pool_attn_kernel<64><<<grid, 128, smem, s>>>(kv, a.ld, a.k_off, a.v_off, a.rows_per_cloud, a.valid_rows, qi, a.partial, tps); break;
  }
  GECCO_CHECK_LAUNCH("pool_attn_kernel");
  const int rows = a.clouds * a.heads * NI;
  pool_combine_kernel<<<ceil_div(rows, 4), 128, 0, s>>>(a.partial, a.heads, a.splits, a.head_dim,
                                                       static_cast<__nv_bfloat16*>(a.out_bf16), a.ldo, rows);
  GECCO_CHECK_LAUNCH("pool_combine_kernel");
  return GECCO_OK;
}

template <int D>
static int launch_unpool_t(const gecco_unpool_args& a, cudaStream_t s) {
  constexpr int smem = 2 * (128 + 2 * NI) * (D + PAD) * 2;
  static bool set = false;
  if (!set) {
    cudaError_t e = cudaFuncSetAttribute(unpool_attn_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(unpool_attn_kernel)");
    set = true;
  }
  dim3 grid(a.rows_per_cloud / 128, a.clouds);
  unpool_attn_kernel<D><<<grid, 256, smem, s>>>(static_cast<const __nv_bfloat16*>(a.q), a.ldq,
                                                static_cast<const __nv_bfloat16*>(a.kv), a.ldkv, a.v_off,
                                                a.rows_per_cloud, a.heads, static_cast<__nv_bfloat16*>(a.out_bf16), a.ldo);
  GECCO_CHECK_LAUNCH("unpool_attn_kernel");
  return GECCO_OK;
}

int launch_unpool_attention(const gecco_unpool_args& a, cudaStream_t s) {
  if (unpool_tc_supported(a)) return launch_unpool_tc(a, s);
  GECCO_REQUIRE(a.inducers == NI, "unpool attention: only 64 inducers are supported (got %d)", a.inducers);
  GECCO_REQUIRE(a.rows_per_cloud % 128 == 0, "unpool attention: rows_per_cloud must be a multiple of 128");
  GECCO_REQUIRE(a.ldq % 8 == 0 && a.ldkv % 8 == 0 && a.ldo % 8 == 0 && a.v_off % 8 == 0, "unpool attention: misaligned layout");
  switch (a.head_dim) {
    case 32: return launch_unpool_t<32>(a, s);
    case 48: return launch_unpool_t<48>(a, s);
    case 64: return launch_unpool_t<64>(a, s);
    default:
      set_error("unpool attention: head_dim must be 32, 48 or 64 (got %d)", a.head_dim);
      return GECCO_ERR_INVALID;
  }
}

}  // namespace gecco

extern "C" int gecco_pool_attention(const gecco_pool_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_pool_attention: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_pool_attention(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_unpool_attention(const gecco_unpool_args* a, void* stream) {
  if (!a) { gecco::set_error("gecco_unpool_attention: null args"); return GECCO_ERR_INVALID; }
  return gecco::launch_unpool_attention(*a, static_cast<cudaStream_t>(stream));
}

extern "C" int gecco_pool_attention_partial(const gecco_pool_args* args, int32_t* splits_used, void* stream) {
  if (args == nullptr || splits_used == nullptr) {
    gecco::set_error("gecco_pool_attention_partial: null args");
    return GECCO_ERR_INVALID;
  }
  int used = 1;
  const int rc = gecco::launch_pool_attention_partial(*args, static_cast<cudaStream_t>(stream), &used);
  *splits_used = used;
  return rc;
}
