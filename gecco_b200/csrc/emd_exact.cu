// Exact earth mover's distance between point clouds of equal size: the optimal assignment, with a certified bound.
//
//   EMD*(X, Y) = min over permutations s of (1/N) sum_i |x_i - y_s(i)|      (Euclidean distance, not its square)
//
// It is what gecco-jax's metrics.py computes with scipy's linear_sum_assignment, and it lies below the approximate
// matching of emd.cu pair by pair.  Method: a forward auction (Bertsekas) with epsilon scaling and Jacobi bidding, one
// 512-thread block per cloud pair.  Persons are the points of the first cloud, objects those of the second; the N x N
// cost matrix is never stored.
//
// Staging.  Both clouds go to shared memory as float4, translated to the bounding-box centre of the pair (of both clouds)
// and multiplied by 2^-e, the power of two that puts the bounding-box diagonal D into [0.5, 1): the auction then runs at
// one scale whatever the units, and the scaling is exact.  Persons carry their object in .w, objects their price.  Beside
// them: owner[N], two bidder lists [N] and one 64-bit bid key per object, 52 N bytes in all (104 KB at 2048 points, two
// blocks per SM; 208 KB at 4096, one).  A cost is recomputed whenever it is needed, always by cost() below:
// c_ij = sqrt(dx^2 + dy^2 + dz^2) in fp32, difference form, IEEE rounding and no contraction, so every use sees the same
// bits.
//
// A round.  Every unassigned person i finds the smallest and second smallest of w_ij = c_ij + p_j over all objects
// (lowest j on equal values) and bids p_j1 + (w2 - w1) + eps on j1, at least the next float above p_j1.  Each object
// keeps the highest bid with a shared 64-bit atomicMax on (bid bits << 32) | (N - 1 - i): prices start at 0 and only
// rise, so bids are non-negative floats whose bits order like integers, and equal bids go to the lowest person.  The
// winner takes the object at its bid, the previous owner is unassigned.  Bids of a round always exceed the object's
// price, i.e. its last winning key, so the keys are never cleared.  A maximum does not depend on arrival order, and a
// bidder's top two values do not depend on how its scan is split (min and max are exact), so results are bitwise
// deterministic.  When fewer bidders than warps remain, the 16 warps split each bidder's scan and merge the top two
// through shared memory: late rounds have only a few bidders, and the number of rounds, not of bids, sets the time.
//
// Schedule.  eps = D/4, D/16, ..., D/4^10 = 2^-20 D: ten phases; prices carry over between phases, assignments reset.
// A phase that needs more than 2^20 rounds (convergence takes a few thousand) stops the pair: it writes NaN to out and
// lower and -1 to match.
//
// Certificate.  After the last phase one more O(N^2) sweep accumulates in double, in a fixed order:
//   upper = (1/N) sum_i c_{i s(i)},   lower = (1/N) (sum_i min_j (c_ij + p_j) - sum_j p_j)   (weak duality);
// on the fp32 costs lower <= OPT <= upper.  eps-complementary slackness bounds upper - lower by eps_final = 2^-20 D, up
// to the rounding of the bids (a few units in the last place of the prices; in practice the gap is far smaller).  upper
// is stored rounded up, lower rounded down.
//
// Cost rounding (u = 2^-24; c the pair's bounding-box centre; R = D/2, so every |p - c| <= R).  Centring rounds each
// coordinate by at most u |p_k - c_k| (the power-of-two scaling is exact), so the difference vector moves by at most
// u (|x - c| + |y - c|) <= 2uR in norm, and its own rounding adds u |x - y|.  The three-term sum of squares is within
// (1 + u)^3 of its value, i.e. the norm within 1.5u + O(u^2), and the square root adds u.  With |x - y| <= 2R:
//     |c_fp32 - |x - y|| <= 2uR + 3.5u |x - y| + O(u^2) <= 9uR + O(u^2) <= 5u D.
// The double sums (N <= 4096 terms) add less than 2^-40 of their size.  Hence, for the true optimum OPT*,
//     lower - 6u D <= OPT* <= upper + 6u D.
// Coordinates must stay below 2^125 in magnitude (the extents must be finite).
#include <math.h>
#include <stdint.h>

#include <algorithm>

#include "common.cuh"

namespace gecco {
namespace {

constexpr int EX_THREADS = 512;
constexpr int EX_WARPS = EX_THREADS / 32;
constexpr int MAX_POINTS = 4096;
constexpr int PHASES = 10;             // eps = D / 4^k, k = 1..10
constexpr int ROUND_CAP = 1 << 20;     // rounds per phase before a pair is given up
constexpr float NO_VALUE = INFINITY;

struct PairMap {
  int mode;  // 0 all pairs, 1 paired, 2 self (upper triangle, mirrored)
  int ma, mb;
};

// Upper-triangle index -> (i, j), i < j, row-major over i (as chamfer.cu).
__device__ __forceinline__ void tri_pair(long long b, int m, int& i, int& j) {
  const double t = 2.0 * m - 1.0;
  long long ii = (long long)floor((t - sqrt(t * t - 8.0 * (double)b)) * 0.5);
  if (ii < 0) ii = 0;
  auto start = [&](long long r) { return r * (2LL * m - r - 1) / 2; };  // first index of row r
  while (ii > 0 && start(ii) > b) --ii;
  while (start(ii + 1) <= b) ++ii;
  i = (int)ii;
  j = (int)(b - start(ii) + ii + 1);
}

// The one cost function: bids and certificate see the same bits.
__device__ __forceinline__ float cost(const float4& p, const float4& q) {
  const float dx = __fsub_rn(p.x, q.x), dy = __fsub_rn(p.y, q.y), dz = __fsub_rn(p.z, q.z);
  return __fsqrt_rn(__fmaf_rn(dz, dz, __fmaf_rn(dy, dy, __fmul_rn(dx, dx))));
}

// Merges (o1, oj, o2) into (w1, j1, w2): smallest value (lowest index on equal values) and second smallest.  Exact, so
// the result does not depend on the order of the merges.
__device__ __forceinline__ void top2_merge(float& w1, int& j1, float& w2, float o1, int oj, float o2) {
  const bool take = o1 < w1 || (o1 == w1 && oj < j1);
  w2 = take ? fminf(o2, w1) : fminf(w2, o1);
  j1 = take ? oj : j1;
  w1 = take ? o1 : w1;
}

__device__ __forceinline__ void top2_warp(float& w1, int& j1, float& w2) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float o1 = __shfl_xor_sync(0xffffffffu, w1, o), o2 = __shfl_xor_sync(0xffffffffu, w2, o);
    const int oj = __shfl_xor_sync(0xffffffffu, j1, o);
    top2_merge(w1, j1, w2, o1, oj, o2);
  }
}

// This lane's share of person pi's scan: objects start, start + stride, ...
__device__ __forceinline__ void scan(const float4& pi, const float4* Q, int n, int start, int stride, float& w1, int& j1,
                                     float& w2) {
  w1 = w2 = NO_VALUE;
  j1 = 0x7fffffff;
  for (int j = start; j < n; j += stride) {
    const float4 q = Q[j];
    const float w = __fadd_rn(cost(pi, q), q.w);
    w2 = fminf(w2, fmaxf(w, w1));
    if (w < w1) j1 = j;
    w1 = fminf(w1, w);
  }
}

// Person i's bid on j1 (one lane): its key goes to the object, j1 to the person's slot.
__device__ __forceinline__ void place_bid(float4* P, const float4* Q, unsigned long long* key, int n, int i, float w1,
                                         int j1, float w2, float eps) {
  const float p = Q[j1].w;
  const float gap = n > 1 ? __fsub_rn(w2, w1) : 0.f;
  const float bid = fmaxf(__fadd_rn(__fadd_rn(p, gap), eps), __uint_as_float(__float_as_uint(p) + 1u));
  atomicMax(&key[j1], (unsigned long long)__float_as_uint(bid) << 32 | (uint32_t)(n - 1 - i));
  P[i].w = __int_as_float(j1);
}

// Fixed-order block sum of one double per thread (butterfly per warp, warps in index order).
__device__ __forceinline__ double block_sum(double v, double* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
  for (int w = 0; w < EX_WARPS; ++w) t += red[w];
  __syncthreads();
  return t;
}

size_t exact_smem_bytes(int n) { return (size_t)n * 52; }

__global__ void __launch_bounds__(EX_THREADS, 2)
    emd_exact_kernel(const float* __restrict__ a, const float* __restrict__ b, int n, PairMap map, float* __restrict__ out,
                     float* __restrict__ lower, int* __restrict__ match) {
  extern __shared__ __align__(16) float4 smem4[];
  __shared__ float bred[EX_WARPS][6];
  __shared__ float tw1[EX_WARPS], tw2[EX_WARPS];
  __shared__ int tj1[EX_WARPS];
  __shared__ double dred[EX_WARPS];
  __shared__ int cnt[2];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long blk = blockIdx.x;
  int i, j;
  long long o1, o2;  // output entries (o2 < 0: none)
  if (map.mode == 0) {
    i = (int)(blk / map.mb);
    j = (int)(blk % map.mb);
    o1 = blk, o2 = -1;
  } else if (map.mode == 1) {
    i = j = (int)blk;
    o1 = blk, o2 = -1;
  } else {
    if (blk < map.ma && tid == 0) {
      out[blk * map.ma + blk] = 0.f;
      if (lower) lower[blk * map.ma + blk] = 0.f;
    }
    if (blk >= (long long)map.ma * (map.ma - 1) / 2) return;
    tri_pair(blk, map.ma, i, j);
    o1 = (long long)i * map.ma + j, o2 = (long long)j * map.ma + i;
  }
  const float* pa = a + (long long)i * n * 3;
  const float* pb = b + (long long)j * n * 3;
  float4* P = smem4;                                                   // [n] persons (a[i]): x, y, z, object
  float4* Q = smem4 + n;                                               // [n] objects (b[j]): x, y, z, price
  unsigned long long* key = reinterpret_cast<unsigned long long*>(Q + n);  // [n] highest bid per object
  int* owner = reinterpret_cast<int*>(key + n);                        // [n]
  int* list0 = owner + n;                                              // [n] bidders, two lists in turn
  int* list1 = list0 + n;

  // bounding box of the pair
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int p = tid; p < 2 * n; p += EX_THREADS) {
    const float* src = p < n ? pa + p * 3 : pb + (p - n) * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = __ldg(src + c);
      lo[c] = fminf(lo[c], v);
      hi[c] = fmaxf(hi[c], v);
    }
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
    for (int c = 0; c < 3; ++c) bred[warp][c] = lo[c], bred[warp][3 + c] = hi[c];
  __syncthreads();
  float ctr[3], ext[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float l = bred[0][c], h = bred[0][3 + c];
    for (int w = 1; w < EX_WARPS; ++w) l = fminf(l, bred[w][c]), h = fmaxf(h, bred[w][3 + c]);
    ctr[c] = 0.5f * (l + h);
    ext[c] = h - l;
  }
  const float emax = fmaxf(ext[0], fmaxf(ext[1], ext[2]));
  if (emax == 0.f) {  // every point of the pair is the same point: cost 0, any permutation
    if (tid == 0) {
      out[o1] = 0.f;
      if (o2 >= 0) out[o2] = 0.f;
      if (lower) {
        lower[o1] = 0.f;
        if (o2 >= 0) lower[o2] = 0.f;
      }
    }
    if (match)
      for (int p = tid; p < n; p += EX_THREADS) match[(long long)i * n + p] = p;
    return;
  }
  // scale 2^-e: the extents to [0.5, 1), then the diagonal to [0.5, 1); both exact
  int e1, e2;
  frexpf(emax, &e1);
  float d2 = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float s = ldexpf(ext[c], -e1);
    d2 = fmaf(s, s, d2);
  }
  const float diag = frexpf(sqrtf(d2), &e2);  // D 2^-e, in [0.5, 1)
  const int e = e1 + e2;
  for (int p = tid; p < n; p += EX_THREADS) {
    P[p] = make_float4(ldexpf(__ldg(pa + p * 3 + 0) - ctr[0], -e), ldexpf(__ldg(pa + p * 3 + 1) - ctr[1], -e),
                       ldexpf(__ldg(pa + p * 3 + 2) - ctr[2], -e), __int_as_float(-1));
    Q[p] = make_float4(ldexpf(__ldg(pb + p * 3 + 0) - ctr[0], -e), ldexpf(__ldg(pb + p * 3 + 1) - ctr[1], -e),
                       ldexpf(__ldg(pb + p * 3 + 2) - ctr[2], -e), 0.f);
    key[p] = 0ull;
  }

  bool failed = false;
#pragma unroll 1
  for (int ph = 1; ph <= PHASES && !failed; ++ph) {
    const float eps = ldexpf(diag, -2 * ph);
    __syncthreads();  // every thread has read the last count of the previous phase
    for (int p = tid; p < n; p += EX_THREADS) owner[p] = -1, list0[p] = p;
    if (tid == 0) cnt[0] = n, cnt[1] = 0;
    __syncthreads();
    int s = 0;
#pragma unroll 1
    for (int rounds = 1;; ++rounds) {
      const int count = cnt[s];
      if (count == 0) break;
      if (rounds > ROUND_CAP) {
        failed = true;
        break;
      }
      const int* cur = s ? list1 : list0;
      int* nxt = s ? list0 : list1;
      float w1, w2;
      int j1;
      if (count >= EX_WARPS) {  // a warp per bidder
        for (int k = warp; k < count; k += EX_WARPS) {
          const int pi = cur[k];
          scan(P[pi], Q, n, lane, 32, w1, j1, w2);
          top2_warp(w1, j1, w2);
          if (lane == 0) place_bid(P, Q, key, n, pi, w1, j1, w2, eps);
        }
      } else {  // g = EX_WARPS / count warps per bidder, merged through shared memory
        const int g = EX_WARPS / count, k = warp / g, sub = warp % g;
        if (k < count) {
          scan(P[cur[k]], Q, n, sub * 32 + lane, g * 32, w1, j1, w2);
          top2_warp(w1, j1, w2);
          if (lane == 0) tw1[warp] = w1, tw2[warp] = w2, tj1[warp] = j1;
        }
        __syncthreads();
        if (warp < count) {
          w1 = w2 = NO_VALUE;
          j1 = 0x7fffffff;
          if (lane < g) w1 = tw1[warp * g + lane], w2 = tw2[warp * g + lane], j1 = tj1[warp * g + lane];
          top2_warp(w1, j1, w2);
          if (lane == 0) place_bid(P, Q, key, n, cur[warp], w1, j1, w2, eps);
        }
      }
      __syncthreads();
      if (tid == 0) cnt[s] = 0;  // every thread has read count; the list is refilled two rounds on
      for (int k = tid; k < count; k += EX_THREADS) {
        const int pi = cur[k];
        const int obj = __float_as_int(P[pi].w);
        const unsigned long long kk = key[obj];
        int loser = pi;
        if ((uint32_t)kk == (uint32_t)(n - 1 - pi)) {  // this round's highest bid on obj is pi's
          loser = owner[obj];
          owner[obj] = pi;
          Q[obj].w = __uint_as_float((uint32_t)(kk >> 32));
        }
        if (loser >= 0) nxt[atomicAdd(&cnt[s ^ 1], 1)] = loser;
      }
      __syncthreads();
      s ^= 1;
    }
  }

  if (failed) {
    if (tid == 0) {
      out[o1] = NAN;
      if (o2 >= 0) out[o2] = NAN;
      if (lower) {
        lower[o1] = NAN;
        if (o2 >= 0) lower[o2] = NAN;
      }
    }
    if (match)
      for (int p = tid; p < n; p += EX_THREADS) match[(long long)i * n + p] = -1;
    return;
  }

  // certificate: the permutation's cost and the dual bound, per thread in point order, then block_sum
  double sc = 0.0, sm = 0.0, sp = 0.0;
  for (int p = tid; p < n; p += EX_THREADS) {
    const float4 pi = P[p];
    const int obj = __float_as_int(pi.w);
    sc += (double)cost(pi, Q[obj]);
    double m = INFINITY;
    for (int q = 0; q < n; ++q) {
      const float4 oq = Q[q];
      m = fmin(m, (double)cost(pi, oq) + (double)oq.w);
    }
    sm += m;
    sp += (double)Q[p].w;
    if (match) match[(long long)i * n + p] = obj;
  }
  sc = block_sum(sc, dred);
  sm = block_sum(sm, dred);
  sp = block_sum(sp, dred);
  if (tid == 0) {
    const float up = __double2float_ru(ldexp(sc / n, e));
    out[o1] = up;
    if (o2 >= 0) out[o2] = up;
    if (lower) {
      const float lw = __double2float_rd(ldexp((sm - sp) / n, e));
      lower[o1] = lw;
      if (o2 >= 0) lower[o2] = lw;
    }
  }
}

}  // namespace
}  // namespace gecco

extern "C" int gecco_emd_exact(const gecco_emd_exact_args* args, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(args != nullptr, "emd_exact: null args");
  const gecco_emd_exact_args& A = *args;
  GECCO_REQUIRE(A.a && A.out, "emd_exact: null argument");
  GECCO_REQUIRE(A.mode == GECCO_CHAMFER_ALL || A.mode == GECCO_CHAMFER_PAIRED || A.mode == GECCO_CHAMFER_SELF,
                "emd_exact: unknown mode %d", A.mode);
  const float* b = A.mode == GECCO_CHAMFER_SELF ? A.a : A.b;
  const int mb = A.mode == GECCO_CHAMFER_SELF ? A.ma : A.mb;
  const int nb = A.mode == GECCO_CHAMFER_SELF ? A.na : A.nb;
  GECCO_REQUIRE(b != nullptr, "emd_exact: null argument");
  GECCO_REQUIRE(A.ma >= 0 && mb >= 0, "emd_exact: negative cloud count");
  GECCO_REQUIRE(A.na == nb, "emd_exact: the clouds of a pair need equal point counts (got %d and %d)", A.na, nb);
  GECCO_REQUIRE(A.na >= 1 && A.na <= MAX_POINTS, "emd_exact: clouds need 1 to %d points (got %d)", MAX_POINTS, A.na);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_PAIRED || A.ma == mb,
                "emd_exact: paired mode needs as many clouds in a as in b (%d, %d)", A.ma, mb);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_SELF || A.b == nullptr || (A.b == A.a && A.mb == A.ma && A.nb == A.na),
                "emd_exact: self mode compares a with itself (b must be NULL or a)");
  GECCO_REQUIRE(A.match == nullptr || A.mode == GECCO_CHAMFER_PAIRED, "emd_exact: match is only written in paired mode");
  long long blocks;
  if (A.mode == GECCO_CHAMFER_ALL)
    blocks = (long long)A.ma * mb;
  else if (A.mode == GECCO_CHAMFER_PAIRED)
    blocks = A.ma;
  else  // the upper triangle; the first ma blocks also write the diagonal
    blocks = std::max<long long>((long long)A.ma * (A.ma - 1) / 2, A.ma);
  if (blocks == 0) return GECCO_OK;
  GECCO_REQUIRE(blocks <= 0x7fffffffLL, "emd_exact: too many cloud pairs (%lld)", blocks);
  const PairMap map{A.mode, A.ma, mb};
  const size_t smem = exact_smem_bytes(A.na);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (smem > 48 * 1024) {  // host-side attribute, no synchronisation
    cudaError_t e = cudaFuncSetAttribute(emd_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail_cuda(e, "emd_exact: shared memory attribute");
  }
  emd_exact_kernel<<<(unsigned)blocks, EX_THREADS, smem, s>>>(A.a, b, A.na, map, A.out, A.lower, A.match);
  GECCO_CHECK_LAUNCH("emd_exact_kernel");
  return GECCO_OK;
}
