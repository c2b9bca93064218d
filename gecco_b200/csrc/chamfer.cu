// Chamfer distance between point clouds: the distance under the 1-NNA / MMD / COV sample-quality metrics
// (gecco_b200/metrics.py; PointFlow's compute_all_metrics protocol, the one GECCO's and its peers' tables use).
//
//   CD(X, Y) = mean_{x in X} min_{y in Y} |x - y|^2  +  mean_{y in Y} min_{x in X} |x - y|^2
//
// One block computes CD for one cloud pair, both directions in ONE pass over the point pairs:
//   - the larger cloud of the pair ("rows") sits in registers, ROWS_PER_LANE points per lane, 2048 rows per pass;
//   - the smaller cloud ("columns") is staged in shared memory as {-2y, |y|^2}, two columns 32 apart packed per 32-byte unit so
//     that a packed FFMA2 computes the distance of one row to two columns;
//   - d = (|x|^2 + |y|^2) + x . (-2y): one FADD2 + three FFMA2 for two pairs (PointFlow's distChamfer expansion);
//   - row minima stay in registers (one FMNMX3 per two pairs);
//   - column minima ride along with the columns: in step s of a 64-column group lane l works on column unit (l + s) mod 32, and
//     the unit's running minimum moves to lane l - 1 with one SHFL, which works on that unit in step s + 1.  After 32 steps a
//     unit's minimum has seen the warp's 256 rows; it is folded into the block's per-column minima in shared memory with an
//     integer atomicMin on the (non-negative) float bits.  A minimum does not depend on the order it is formed in, so the
//     result is exact whatever order the warps arrive in;
//   - the two directional sums are formed in a fixed order (per lane, butterfly per warp, warps in index order, passes in
//     order, in double from the warp level on): the result is bitwise deterministic.
// Both clouds are translated by the bounding-box centre of the first cloud of the pair while they are staged: distances do
// not change and |x|^2 + |y|^2 - 2 x.y does not cancel away the digits of clouds that sit far from the origin.
//
// Pair modes (block -> pair map, same per-pair code): all pairs a x b; paired (i, i); self (b is a): upper triangle, mirrored,
// diagonal exactly 0.  Tails of any point count are handled inside (rows / columns past the end are +inf).
#include <math.h>

#include "common.cuh"

namespace gecco {
namespace {

constexpr int CH_THREADS = 256;
constexpr int CH_WARPS = CH_THREADS / 32;
constexpr int ROWS_PER_LANE = 8;
constexpr int ROWS_PER_PASS = CH_THREADS * ROWS_PER_LANE;  // 2048
constexpr int TILE_COLS = 2048;                            // columns staged per shared-memory tile (32 KB)
constexpr int GROUP_COLS = 64;                             // columns swept by a warp in one 32-step rotation
constexpr int MAX_SMALL_POINTS = 32768;                    // per-column minima of the smaller cloud live in shared memory

__device__ __forceinline__ float min3f(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// +0 for anything not positive (also -0 and rounding below zero): the bit patterns then order like the values
__device__ __forceinline__ float clamp0(float v) { return v > 0.f ? v : 0.f; }

struct PairMap {
  int mode;  // 0 all pairs, 1 paired, 2 self (upper triangle)
  int ma, mb;
};

// Upper-triangle index -> (i, j), i < j, row-major over i.
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

__global__ void __launch_bounds__(CH_THREADS, 2) chamfer_kernel(const float* __restrict__ a, int na, const float* __restrict__ b,
                                                                int nb, PairMap map, int swap, float* __restrict__ out) {
  extern __shared__ __align__(16) float smem[];
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
    if (blk >= (long long)map.ma * (map.ma - 1) / 2) return;
    tri_pair(blk, map.ma, i, j);
  }
  const float* pa = a + (long long)i * na * 3;
  const float* pb = b + (long long)j * nb * 3;
  // rows: the larger cloud (registers); cols: the smaller one (shared memory)
  const float* rows = swap ? pb : pa;
  const float* cols = swap ? pa : pb;
  const int nrow = swap ? nb : na, ncol = swap ? na : nb;
  const int ncol_pad = (ncol + GROUP_COLS - 1) / GROUP_COLS * GROUP_COLS;
  const int tile_cols = min(ncol_pad, TILE_COLS);

  float* tile = smem;                                             // [tile_cols / 2 units][8]
  int* colmin = reinterpret_cast<int*>(smem + tile_cols * 4);     // [ncol_pad] float bits
  float* red = reinterpret_cast<float*>(colmin + ncol_pad);       // [CH_WARPS][6] bounding box partials
  double* dred = reinterpret_cast<double*>(red + CH_WARPS * 6 + 2);  // [CH_WARPS]; +2 floats keep 8-byte alignment

  // bounding-box centre of the first cloud of the pair
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int p = tid; p < na; p += CH_THREADS)
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
  for (int p = tid; p < ncol_pad; p += CH_THREADS) colmin[p] = __float_as_int(INFINITY);
  __syncthreads();
  float ctr[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float l = red[c], h = red[3 + c];
    for (int w = 1; w < CH_WARPS; ++w) l = fminf(l, red[w * 6 + c]), h = fmaxf(h, red[w * 6 + 3 + c]);
    ctr[c] = 0.5f * (l + h);
  }

  double row_sum = 0.0;  // meaningful in thread 0 only
  const bool one_tile = ncol_pad <= TILE_COLS;
  auto stage = [&](int col0) {  // columns [col0, col0 + tile_cols) -> tile; pads: y = 0, |y|^2 = +inf
    for (int c = tid; c < tile_cols; c += CH_THREADS) {
      const int col = col0 + c;
      float y0 = 0.f, y1 = 0.f, y2 = 0.f, n = INFINITY;
      if (col < ncol) {
        y0 = __ldg(cols + col * 3 + 0) - ctr[0];
        y1 = __ldg(cols + col * 3 + 1) - ctr[1];
        y2 = __ldg(cols + col * 3 + 2) - ctr[2];
        n = fmaf(y2, y2, fmaf(y1, y1, y0 * y0));
      }
      // unit u of group g holds columns g*64 + u (even slot) and g*64 + 32 + u (odd slot)
      const int g = c / GROUP_COLS, r = c % GROUP_COLS, u = r & 31, hi_slot = r >> 5;
      float* t = tile + (g * 32 + u) * 8 + hi_slot;
      t[0] = -2.f * y0;
      t[2] = -2.f * y1;
      t[4] = -2.f * y2;
      t[6] = n;
    }
  };
  if (one_tile) stage(0);  // the whole smaller cloud stays resident across the row passes

  for (int row0 = 0; row0 < nrow; row0 += ROWS_PER_PASS) {
    float2 xx[ROWS_PER_LANE], xy[ROWS_PER_LANE], xz[ROWS_PER_LANE], xn[ROWS_PER_LANE];
    float rmin[ROWS_PER_LANE];
    const int wrow0 = row0 + warp * 32 * ROWS_PER_LANE;
    const bool warp_live = wrow0 < nrow;  // warp-uniform: warps past the end of the rows skip the sweep
#pragma unroll
    for (int r = 0; r < ROWS_PER_LANE; ++r) {
      const int row = wrow0 + r * 32 + lane;
      float x0 = 0.f, x1 = 0.f, x2 = 0.f, n = INFINITY;
      if (row < nrow) {
        x0 = __ldg(rows + row * 3 + 0) - ctr[0];
        x1 = __ldg(rows + row * 3 + 1) - ctr[1];
        x2 = __ldg(rows + row * 3 + 2) - ctr[2];
        n = fmaf(x2, x2, fmaf(x1, x1, x0 * x0));
      }
      xx[r] = make_float2(x0, x0);
      xy[r] = make_float2(x1, x1);
      xz[r] = make_float2(x2, x2);
      xn[r] = make_float2(n, n);
      rmin[r] = INFINITY;
    }
    for (int col0 = 0; col0 < ncol_pad; col0 += TILE_COLS) {
      if (!one_tile) {
        __syncthreads();  // the previous tile is no longer read
        stage(col0);
      }
      __syncthreads();
      const int tcols = min(TILE_COLS, ncol_pad - col0);
      if (warp_live) {
        for (int g = 0; g < tcols / GROUP_COLS; ++g) {
          const float4* unit = reinterpret_cast<const float4*>(tile + g * 32 * 8);
          float c0 = INFINITY, c1 = INFINITY;  // running minima of the unit this lane works on (even / odd slot)
#pragma unroll 4
          for (int s = 0; s < 32; ++s) {
            const int u = (lane + s) & 31;
            const float4 p = unit[u * 2], q = unit[u * 2 + 1];
            const float2 yx = make_float2(p.x, p.y), yy = make_float2(p.z, p.w);
            const float2 yz = make_float2(q.x, q.y), yn = make_float2(q.z, q.w);
            float2 d[ROWS_PER_LANE];
#pragma unroll
            for (int r = 0; r < ROWS_PER_LANE; ++r) {
              d[r] = __fadd2_rn(xn[r], yn);
              d[r] = __ffma2_rn(xx[r], yx, d[r]);
              d[r] = __ffma2_rn(xy[r], yy, d[r]);
              d[r] = __ffma2_rn(xz[r], yz, d[r]);
              rmin[r] = min3f(rmin[r], d[r].x, d[r].y);
            }
#pragma unroll
            for (int r = 0; r < ROWS_PER_LANE; r += 2) {
              c0 = min3f(c0, d[r].x, d[r + 1].x);
              c1 = min3f(c1, d[r].y, d[r + 1].y);
            }
            if (s != 31) {
              c0 = __shfl_sync(0xffffffffu, c0, (lane + 1) & 31);
              c1 = __shfl_sync(0xffffffffu, c1, (lane + 1) & 31);
            }
          }
          const int u = (lane + 31) & 31;  // the unit whose minimum this lane holds after the last step
          atomicMin(&colmin[col0 + g * GROUP_COLS + u], __float_as_int(clamp0(c0)));
          atomicMin(&colmin[col0 + g * GROUP_COLS + 32 + u], __float_as_int(clamp0(c1)));
        }
      }
    }
    // row minima of this pass -> one sum, in a fixed order
    float s = 0.f;
#pragma unroll
    for (int r = 0; r < ROWS_PER_LANE; ++r)
      if (wrow0 + r * 32 + lane < nrow) s += clamp0(rmin[r]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) dred[warp] = (double)s;
    __syncthreads();
    if (tid == 0)
      for (int w = 0; w < CH_WARPS; ++w) row_sum += dred[w];
    __syncthreads();
  }

  // column minima -> one sum, in a fixed order
  float s = 0.f;
  for (int c = tid; c < ncol; c += CH_THREADS) s += __int_as_float(colmin[c]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) dred[warp] = (double)s;
  __syncthreads();
  if (tid == 0) {
    double col_sum = 0.0;
    for (int w = 0; w < CH_WARPS; ++w) col_sum += dred[w];
    const float cd = (float)(row_sum / nrow + col_sum / ncol);
    if (map.mode == 0) {
      out[blk] = cd;
    } else if (map.mode == 1) {
      out[i] = cd;
    } else {
      out[(long long)i * map.ma + j] = cd;
      out[(long long)j * map.ma + i] = cd;
    }
  }
}

size_t chamfer_smem_bytes(int ncol) {
  const int ncol_pad = (ncol + GROUP_COLS - 1) / GROUP_COLS * GROUP_COLS;
  const int tile_cols = ncol_pad < TILE_COLS ? ncol_pad : TILE_COLS;
  return (size_t)tile_cols * 16 + (size_t)ncol_pad * 4 + (CH_WARPS * 6 + 2) * 4 + CH_WARPS * 8;
}

}  // namespace
}  // namespace gecco

extern "C" int gecco_chamfer(const gecco_chamfer_args* args, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(args != nullptr, "chamfer: null args");
  const gecco_chamfer_args& A = *args;
  GECCO_REQUIRE(A.a && A.out, "chamfer: null argument");
  GECCO_REQUIRE(A.mode == GECCO_CHAMFER_ALL || A.mode == GECCO_CHAMFER_PAIRED || A.mode == GECCO_CHAMFER_SELF,
                "chamfer: unknown mode %d", A.mode);
  const float* b = A.mode == GECCO_CHAMFER_SELF ? A.a : A.b;
  const int mb = A.mode == GECCO_CHAMFER_SELF ? A.ma : A.mb;
  const int nb = A.mode == GECCO_CHAMFER_SELF ? A.na : A.nb;
  GECCO_REQUIRE(b != nullptr, "chamfer: null argument");
  GECCO_REQUIRE(A.ma >= 0 && mb >= 0, "chamfer: negative cloud count");
  GECCO_REQUIRE(A.na >= 1 && nb >= 1, "chamfer: clouds need at least one point (got %d and %d)", A.na, nb);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_PAIRED || A.ma == mb, "chamfer: paired mode needs as many clouds in a as in b (%d, %d)",
                A.ma, mb);
  GECCO_REQUIRE(A.mode != GECCO_CHAMFER_SELF || A.b == nullptr || (A.b == A.a && A.mb == A.ma && A.nb == A.na),
                "chamfer: self mode compares a with itself (b must be NULL or a)");
  const int small = A.na < nb ? A.na : nb;
  GECCO_REQUIRE(small <= MAX_SMALL_POINTS, "chamfer: the smaller cloud of a pair may have at most %d points (got %d and %d)",
                MAX_SMALL_POINTS, A.na, nb);
  long long blocks;
  if (A.mode == GECCO_CHAMFER_ALL)
    blocks = (long long)A.ma * mb;
  else if (A.mode == GECCO_CHAMFER_PAIRED)
    blocks = A.ma;
  else
    blocks = A.ma > 2 ? (long long)A.ma * (A.ma - 1) / 2 : A.ma;  // the first ma blocks also write the diagonal
  if (blocks == 0) return GECCO_OK;
  GECCO_REQUIRE(blocks <= 0x7fffffffLL, "chamfer: too many cloud pairs (%lld)", blocks);
  const int swap = nb > A.na ? 1 : 0;  // the smaller cloud goes to shared memory
  const size_t smem = chamfer_smem_bytes(swap ? A.na : nb);
  if (smem > 48 * 1024) {  // only clouds past ~8k points on both sides (host-side attribute, no synchronisation)
    cudaError_t e = cudaFuncSetAttribute(chamfer_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail_cuda(e, "chamfer: shared memory attribute");
  }
  PairMap map{A.mode, A.ma, mb};
  chamfer_kernel<<<(unsigned)blocks, CH_THREADS, smem, static_cast<cudaStream_t>(stream)>>>(A.a, A.na, b, nb, map, swap, A.out);
  GECCO_CHECK_LAUNCH("chamfer_kernel");
  return GECCO_OK;
}
