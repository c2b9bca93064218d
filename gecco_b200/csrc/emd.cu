// Approximate earth mover's distance (EMD) between point clouds of equal size: the second distance of the 1-NNA / MMD /
// COV sample-quality metrics (gecco_b200/metrics.py).  It is the approximate matching of Fan et al. 2017 ("approxmatch" /
// "match_cost" in PSGN and PointFlow's StructuralLosses) divided by N, as in PointFlow's emd_approx.  It is not the optimal
// transport cost.  With d2[k,l] = |x_k - y_l|^2, dist = sqrt(d2), remL = remR = 1, cost = 0:
//
//   for j = 7, 6, ..., 0, -1, -2:   level = -4^j (0 for j = -2), e = exp(level * d2)
//     ratioL[k] = remL[k] / (1e-9 + sum_l e[k,l] remR[l])                         pass 1 (rows)
//     sumr[l]   = remR[l] sum_k e[k,l] ratioL[k]                                    pass 2 (columns)
//     ratioR[l] = min(remR[l] / (sumr[l] + 1e-9), 1) remR[l];  remR[l] = max(0, remR[l] - sumr[l])
//     w[k,l] = e[k,l] ratioL[k] ratioR[l];  remL[k] = max(0, remL[k] - sum_l w[k,l]);  cost += sum w dist   pass 3 (rows)
//   EMD(X, Y) = cost / N
//
// One 256-thread block per cloud pair; X ("rows") and Y ("columns") are staged in shared memory as float4 {x, y, z, ratio},
// plus remR.  A thread owns R rows (row sweeps) and the R columns of the same indices (column sweeps); every other point
// is a broadcast shared-memory load that serves all R owned points.  The match matrix is never stored:
//   - pass 3 of level j and pass 1 of level j - 1 are ONE row sweep (pass 1 needs the updated remR, and the updated remL
//     only once the row is done).  It evaluates e_{j-1} = exp(-4^{j-1} d2) with one ex2 and gets e_j = e_{j-1}^4 with two
//     multiplications, so a point pair costs one ex2 and one sqrt;
//   - at level 0 e = 1: the column sweep is O(N) and the last row sweep needs only the sqrt.
// That is 20 O(N^2) sweeps and 29 MUFU operations per point pair.
// exp(-4^j d2) = ex2(-|s x - s y|^2) with s = 2^j sqrt(log2 e): the staged coordinates carry that scale, and going one level
// down halves them (exact).  dist = |s x - s y| / s.  Before the scaling both clouds are translated by the bounding-box
// centre of X, and d2 is formed from coordinate differences: the level -4^7 multiplies absolute errors of d2 by 16384, so
// the |x|^2 + |y|^2 - 2 x.y expansion of chamfer.cu would not do.
// Every sum has a fixed order (per thread in point order, then butterfly per warp, warps in index order in double): the
// result is bitwise deterministic and does not depend on which mode computed it.
#include <math.h>

#include "common.cuh"

namespace gecco {
namespace {

constexpr int EMD_THREADS = 256;
constexpr int EMD_WARPS = EMD_THREADS / 32;
constexpr int MAX_POINTS = 4096;
constexpr float SQRT_LOG2E = 1.20112240878644983f;
constexpr float INV_SQRT_LOG2E = 0.83255461115769776f;

// 2^-x and sqrt(x), one MUFU instruction each
__device__ __forceinline__ float ex2_neg(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(-x));
  return y;
}
__device__ __forceinline__ float sqrt_mufu(float x) {
  float y;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ float sq_dist(float x, float y, float z, const float4& q) {
  const float dx = x - q.x, dy = y - q.y, dz = z - q.z;
  return fmaf(dz, dz, fmaf(dy, dy, dx * dx));
}

enum RowSweep {
  ROW_FIRST,       // pass 1 of level 7 (remR = 1)
  ROW_FUSED,       // pass 3 of level j >= 0 with pass 1 of level j - 1; rows are halved to the scale of level j - 1
  ROW_FUSED_LAST,  // pass 3 of level -1 with pass 1 of level 0 (e = 1: sum_l remR[l], the same for every row)
  ROW_FINAL,       // pass 3 of level 0 (e = 1): cost only
};

// Rows k = r * 256 + tid of P against every column of Q.  inv_s: 1 / the coordinate scale, for the cost.
template <int R, int KIND>
__device__ __forceinline__ void row_sweep(float4* P, const float4* Q, const float* remR, int n, float (&remL)[R],
                                          float inv_s, float& cost) {
  const int tid = threadIdx.x;
  float px[R], py[R], pz[R], aw[R], ac[R], an[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int k = r * EMD_THREADS + tid;
    float4 p = k < n ? P[k] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float h = KIND == ROW_FUSED ? 0.5f : 1.f;
    px[r] = p.x * h, py[r] = p.y * h, pz[r] = p.z * h;
    aw[r] = ac[r] = an[r] = 0.f;
  }
  float tot = 0.f;  // ROW_FUSED_LAST: sum_l remR[l]
  if ((tid & ~31) < n) {  // warps without a valid row skip the sweep
#pragma unroll 2
    for (int l = 0; l < n; ++l) {
      const float4 q = Q[l];
      float rr = 0.f;
      if (KIND == ROW_FUSED) rr = remR[l];
      if (KIND == ROW_FUSED_LAST) tot += remR[l];
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const float d2 = sq_dist(px[r], py[r], pz[r], q);
        if (KIND == ROW_FIRST) {
          an[r] += ex2_neg(d2);
        } else if (KIND == ROW_FUSED) {
          const float e1 = ex2_neg(d2);  // level j - 1
          const float e2 = e1 * e1;
          const float t = (e2 * e2) * q.w;  // e_j ratioR[l]
          aw[r] += t;
          ac[r] = fmaf(t, sqrt_mufu(d2), ac[r]);
          an[r] = fmaf(e1, rr, an[r]);
        } else if (KIND == ROW_FUSED_LAST) {
          const float t = ex2_neg(d2) * q.w;
          aw[r] += t;
          ac[r] = fmaf(t, sqrt_mufu(d2), ac[r]);
        } else {
          ac[r] = fmaf(q.w, sqrt_mufu(d2), ac[r]);
        }
      }
    }
  }
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int k = r * EMD_THREADS + tid;
    if (k >= n) continue;
    if (KIND == ROW_FIRST) {
      P[k].w = 1.f / (1e-9f + an[r]);
    } else {
      const float rl = P[k].w;
      cost += rl * ac[r] * inv_s;
      if (KIND != ROW_FINAL) {
        remL[r] = fmaxf(0.f, remL[r] - rl * aw[r]);
        P[k] = make_float4(px[r], py[r], pz[r], remL[r] / (1e-9f + (KIND == ROW_FUSED ? an[r] : tot)));
      }
    }
  }
}

// Pass 2 for columns l = r * 256 + tid: ratioR -> Q[l].w, remR updated; LEVEL0: e = 1.  halve: move the columns to the
// scale of the next level.
template <int R, bool LEVEL0>
__device__ __forceinline__ void col_sweep(const float4* P, float4* Q, float* remR, int n, bool halve) {
  const int tid = threadIdx.x;
  float qx[R], qy[R], qz[R], acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int l = r * EMD_THREADS + tid;
    const float4 q = l < n ? Q[l] : make_float4(0.f, 0.f, 0.f, 0.f);
    qx[r] = q.x, qy[r] = q.y, qz[r] = q.z;
    acc[r] = 0.f;
  }
  if (LEVEL0) {  // sum_k ratioL[k], the same for every column (every thread forms it in the same order)
    float s[4] = {0.f, 0.f, 0.f, 0.f};
    int k = 0;
    for (; k + 4 <= n; k += 4)
#pragma unroll
      for (int u = 0; u < 4; ++u) s[u] += P[k + u].w;
    for (; k < n; ++k) s[0] += P[k].w;
    const float t = (s[0] + s[1]) + (s[2] + s[3]);
#pragma unroll
    for (int r = 0; r < R; ++r) acc[r] = t;
  } else if ((tid & ~31) < n) {
#pragma unroll 2
    for (int k = 0; k < n; ++k) {
      const float4 p = P[k];
#pragma unroll
      for (int r = 0; r < R; ++r) acc[r] = fmaf(ex2_neg(sq_dist(qx[r], qy[r], qz[r], p)), p.w, acc[r]);
    }
  }
  const float h = halve ? 0.5f : 1.f;
#pragma unroll
  for (int r = 0; r < R; ++r) {
    const int l = r * EMD_THREADS + tid;
    if (l >= n) continue;
    const float rr = remR[l];
    const float sumr = rr * acc[r];
    remR[l] = fmaxf(0.f, rr - sumr);
    Q[l] = make_float4(qx[r] * h, qy[r] * h, qz[r] * h, fminf(rr / (sumr + 1e-9f), 1.f) * rr);
  }
}

struct PairMap {
  int mode;  // 0 all pairs, 1 paired, 2 self (ordered pairs i != j)
  int ma, mb;
};

size_t emd_smem_bytes(int n) { return (size_t)n * 36 + EMD_WARPS * 8 + EMD_WARPS * 6 * 4; }

template <int R>
__global__ void __launch_bounds__(EMD_THREADS, R <= 8 ? 3 : 1)
    emd_kernel(const float* __restrict__ a, const float* __restrict__ b, int n, PairMap map, float* __restrict__ out) {
  extern __shared__ __align__(16) float4 smem4[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long blk = blockIdx.x;
  int i, j;
  if (map.mode == 0) {
    i = (int)(blk / map.mb);
    j = (int)(blk % map.mb);
  } else if (map.mode == 1) {
    i = j = (int)blk;
  } else {
    if (blk < map.ma && tid == 0) out[blk * map.ma + blk] = 0.f;
    if (blk >= (long long)map.ma * (map.ma - 1)) return;
    i = (int)(blk / (map.ma - 1));
    j = (int)(blk % (map.ma - 1));
    j += j >= i;
  }
  const float* pa = a + (long long)i * n * 3;
  const float* pb = b + (long long)j * n * 3;
  float4* P = smem4;                                        // [n] rows (X = a[i])
  float4* Q = smem4 + n;                                    // [n] columns (Y = b[j])
  double* dred = reinterpret_cast<double*>(smem4 + 2 * n);  // [EMD_WARPS]
  float* red = reinterpret_cast<float*>(dred + EMD_WARPS);  // [EMD_WARPS][6] bounding-box partials
  float* remR = red + EMD_WARPS * 6;                        // [n]

  // bounding-box centre of X
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int p = tid; p < n; p += EMD_THREADS)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = __ldg(pa + p * 3 + c);
      lo[c] = fminf(lo[c], v);
      hi[c] = fmaxf(hi[c], v);
    }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      lo[c] = fminf(lo[c], __shfl_xor_sync(0xffffffffu, lo[c], o));
      hi[c] = fmaxf(hi[c], __shfl_xor_sync(0xffffffffu, hi[c], o));
    }
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 3; ++c) red[warp * 6 + c] = lo[c], red[warp * 6 + 3 + c] = hi[c];
  __syncthreads();
  float ctr[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float l = red[c], h = red[3 + c];
    for (int w = 1; w < EMD_WARPS; ++w) l = fminf(l, red[w * 6 + c]), h = fmaxf(h, red[w * 6 + 3 + c]);
    ctr[c] = 0.5f * (l + h);
  }
  const float s7 = 128.f * SQRT_LOG2E;  // scale of level 7
  for (int p = tid; p < n; p += EMD_THREADS) {
    P[p] = make_float4((__ldg(pa + p * 3 + 0) - ctr[0]) * s7, (__ldg(pa + p * 3 + 1) - ctr[1]) * s7,
                       (__ldg(pa + p * 3 + 2) - ctr[2]) * s7, 0.f);
    Q[p] = make_float4((__ldg(pb + p * 3 + 0) - ctr[0]) * s7, (__ldg(pb + p * 3 + 1) - ctr[1]) * s7,
                       (__ldg(pb + p * 3 + 2) - ctr[2]) * s7, 0.f);
    remR[p] = 1.f;
  }
  float remL[R];
#pragma unroll
  for (int r = 0; r < R; ++r) remL[r] = 1.f;
  float cost = 0.f;
  __syncthreads();

  row_sweep<R, ROW_FIRST>(P, Q, remR, n, remL, 0.f, cost);
  __syncthreads();
#pragma unroll 1
  for (int lv = 7; lv >= 0; --lv) {
    col_sweep<R, false>(P, Q, remR, n, true);
    __syncthreads();
    row_sweep<R, ROW_FUSED>(P, Q, remR, n, remL, ldexpf(INV_SQRT_LOG2E, 1 - lv), cost);
    __syncthreads();
  }
  // level -1: the coordinates stay at its scale (2^-1 sqrt(log2 e)) for the rest
  const float inv_s = 2.f * INV_SQRT_LOG2E;
  col_sweep<R, false>(P, Q, remR, n, false);
  __syncthreads();
  row_sweep<R, ROW_FUSED_LAST>(P, Q, remR, n, remL, inv_s, cost);
  __syncthreads();
  col_sweep<R, true>(P, Q, remR, n, false);
  __syncthreads();
  row_sweep<R, ROW_FINAL>(P, Q, remR, n, remL, inv_s, cost);

#pragma unroll
  for (int o = 16; o > 0; o >>= 1) cost += __shfl_xor_sync(0xffffffffu, cost, o);
  if (lane == 0) dred[warp] = (double)cost;
  __syncthreads();
  if (tid == 0) {
    double total = 0.0;
    for (int w = 0; w < EMD_WARPS; ++w) total += dred[w];
    const float emd = (float)(total / n);
    if (map.mode == 0)
      out[blk] = emd;
    else if (map.mode == 1)
      out[i] = emd;
    else
      out[(long long)i * map.ma + j] = emd;
  }
}

template <int R>
int launch(const float* a, const float* b, int n, PairMap map, long long blocks, float* out, cudaStream_t stream) {
  const size_t smem = emd_smem_bytes(n);
  if (smem > 48 * 1024) {  // host-side attribute, no synchronisation
    cudaError_t e = cudaFuncSetAttribute(emd_kernel<R>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail_cuda(e, "emd: shared memory attribute");
  }
  emd_kernel<R><<<(unsigned)blocks, EMD_THREADS, smem, stream>>>(a, b, n, map, out);
  GECCO_CHECK_LAUNCH("emd_kernel");
  return GECCO_OK;
}

}  // namespace
}  // namespace gecco

extern "C" int gecco_emd(const gecco_chamfer_args* args, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(args != nullptr, "emd: null args");
  const gecco_chamfer_args& A = *args;
  GECCO_REQUIRE(A.a && A.out, "emd: null argument");
  GECCO_REQUIRE(A.mode == GECCO_CHAMFER_ALL || A.mode == GECCO_CHAMFER_PAIRED || A.mode == GECCO_CHAMFER_SELF,
                "emd: unknown mode %d", A.mode);
  const float* b = A.mode == GECCO_CHAMFER_SELF ? A.a : A.b;
  const int mb = A.mode == GECCO_CHAMFER_SELF ? A.ma : A.mb;
  const int nb = A.mode == GECCO_CHAMFER_SELF ? A.na : A.nb;
  GECCO_REQUIRE(b != nullptr, "emd: null argument");
  GECCO_REQUIRE(A.ma >= 0 && mb >= 0, "emd: negative cloud count");
  GECCO_REQUIRE(A.na == nb, "emd: the clouds of a pair need equal point counts (got %d and %d)", A.na, nb);
  GECCO_REQUIRE(A.na >= 1 && A.na <= MAX_POINTS, "emd: clouds need 1 to %d points (got %d)", MAX_POINTS, A.na);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_PAIRED || A.ma == mb, "emd: paired mode needs as many clouds in a as in b (%d, %d)",
                A.ma, mb);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_SELF || A.b == nullptr || (A.b == A.a && A.mb == A.ma && A.nb == A.na),
                "emd: self mode compares a with itself (b must be NULL or a)");
  long long blocks;
  if (A.mode == GECCO_CHAMFER_ALL)
    blocks = (long long)A.ma * mb;
  else if (A.mode == GECCO_CHAMFER_PAIRED)
    blocks = A.ma;
  else
    blocks = A.ma >= 2 ? (long long)A.ma * (A.ma - 1) : A.ma;  // the first ma blocks also write the diagonal
  if (blocks == 0) return GECCO_OK;
  GECCO_REQUIRE(blocks <= 0x7fffffffLL, "emd: too many cloud pairs (%lld)", blocks);
  const PairMap map{A.mode, A.ma, mb};
  const int n = A.na;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // R owned rows (and columns) per thread: the smallest power of two with 256 R >= n
  if (n <= 256) return launch<1>(A.a, b, n, map, blocks, A.out, s);
  if (n <= 512) return launch<2>(A.a, b, n, map, blocks, A.out, s);
  if (n <= 1024) return launch<4>(A.a, b, n, map, blocks, A.out, s);
  if (n <= 2048) return launch<8>(A.a, b, n, map, blocks, A.out, s);
  return launch<16>(A.a, b, n, map, blocks, A.out, s);
}
