// Nearest neighbours between paired point clouds, both directions, as indices and squared distances: the per-point
// numbers under the F-score and the paired Chamfer distance of conditional reconstructions (gecco_b200/metrics.py).
//
//   idx_xy[b, i] = argmin_j |x_bi - y_bj|^2   (lowest j on ties),   dist_xy[b, i] = |x_bi - y_b,idx|^2;   y -> x likewise.
//
// Three launches and a memset on the caller's stream:
//   1. keys <- all ones (cudaMemsetAsync);
//   2. centre_kernel: per pair the bounding-box centre c of x_b, once (not once per block);
//   3. nearest_kernel: grid (pair, row tile, column chunk).  x is the row side: 2048 rows per block in registers, 8 per
//      lane.  A chunk of y (128 to 2048 columns) is staged in shared memory as {-2y, |y|^2}, two columns 32 apart per
//      32-byte unit, exactly as in chamfer.cu, after both clouds are translated by c.  d = (|x|^2 + |y|^2) + x.(-2y) is
//      one FADD2 and three FFMA2 for two point pairs.  Both directions come out of the same pass:
//        - row side: d's float bits with the sign cleared and the low 6 bits replaced by the column's position in its
//          64-column group form a key; one FMNMX3 per two pairs keeps the minimum key of each row over the group.  Once
//          per group it becomes a 64-bit key ((value bits) << 32 | column) and lowers the row's running minimum, which
//          the row's own thread keeps in shared memory;
//        - column side: the same bits with the low 8 bits replaced by the row's position in its warp (256 rows) form a
//          second key.  Column keys ride along with their columns around the warp as in chamfer.cu (one SHFL per unit
//          and step); after 32 steps a key has seen the warp's 256 rows and is folded into the block's per-column
//          minimum in shared memory with a 64-bit atomicMin on ((value bits) << 32 | row);
//        - at the end of the block every row and every column does one 64-bit atomicMin of its key into global scratch.
//      A key's value bits are the non-negative |d| with its low bits cut off, and a 64-bit integer minimum then takes
//      the smallest value first and the lowest index on equal values.  A minimum does not depend on arrival order or on
//      how the grid is cut into blocks, so the result is bitwise deterministic;
//   4. finish_kernel: per point, decode the index and recompute the distance in difference form from the caller's
//      coordinates, (p - q).(p - q) in fp32.
//
// Error bound (u = 2^-24; c the bounding-box centre of x_b; R the largest |p - c| over the points p of x_b and y_b;
// d* the exact minimum over the candidates of a point): the reported distance d satisfies
//     d* (1 - 5u) <= d <= d* + B,   B = 2^-13 d* + 72 u R^2.
// Derivation.  For a query p and a candidate q with a = |p - c|, b = |q - c|, the search value s(p, q) is computed on the
// rounded centred coordinates (each off by at most u |p_k - c_k|, u |q_k - c_k|: |p - q|^2 moves by at most
// 2u (a + b)^2), with the norms from two FMAs and an FMUL (at most 3u a^2, 3u b^2) and the expansion from one FADD and
// three FMAs (at most 4u (a^2 + b^2 + 2ab), |p.q| <= ab): |s - |p - q|^2| <= 9u (a + b)^2 <= 36 u R^2 =: E.  The keys
// compare |s| with the low k bits cut (k = 6 rows, 8 columns), which lowers a value by at most 2^-15 of it.  The chosen
// candidate therefore has |p - q|^2 <= (d* + E) / (1 - 2^-15) + E, i.e. at most 2^-14 d* + 2E + O(u^2) above d*, and
// the difference form adds at most 5u of its own value.  Wherever the second nearest candidate lies more than B above the
// nearest, the index is the exact argmin.  Coordinates must stay below ~1e18 in magnitude (|p - c|^2 must be finite).
#include <math.h>
#include <stdint.h>

#include "common.cuh"

namespace gecco {
namespace {

constexpr int NN_THREADS = 256;
constexpr int NN_WARPS = NN_THREADS / 32;
constexpr int ROWS_PER_LANE = 8;
constexpr int ROWS_PER_TILE = NN_THREADS * ROWS_PER_LANE;  // 2048
constexpr int GROUP_COLS = 64;                             // columns swept by a warp in one 32-step rotation
constexpr int MAX_CHUNK = 2048;                            // columns per block: 32 KB tile + 16 KB column keys + 16 KB row keys
constexpr int MIN_CHUNK = 128;
constexpr int MAX_POINTS = 1 << 24;
constexpr float PAD_NORM = 1e38f;          // |p|^2 of padding rows and columns: finite, larger than any real distance
constexpr uint32_t ROW_MASK = 0x7fffffc0u;  // sign cleared, low 6 bits: column within the 64-column group
constexpr uint32_t COL_MASK = 0x7fffff00u;  // sign cleared, low 8 bits: row within the warp's 256 rows
constexpr unsigned long long NO_KEY = ~0ull;

__device__ __forceinline__ float min3f(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// (d & mask) | id, as a float: non-negative, so float order is the order of the bits (denormals included: no .ftz).
// One LOP3; written in PTX because the compiler otherwise splits it in two when it can see the bits of id.
template <uint32_t MASK>
__device__ __forceinline__ float key32(float d, uint32_t id) {
  uint32_t k;
  asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(k) : "r"(__float_as_uint(d)), "n"(MASK), "r"(id));
  return __uint_as_float(k);
}

__global__ void __launch_bounds__(NN_THREADS) centre_kernel(const float* __restrict__ x, int nx, float* __restrict__ ctr) {
  __shared__ float red[NN_WARPS][6];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const float* px = x + (long long)blockIdx.x * nx * 3;
  float lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
  for (int p = tid; p < nx; p += NN_THREADS)
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v = __ldg(px + (long long)p * 3 + c);
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
    for (int c = 0; c < 3; ++c) red[warp][c] = lo[c], red[warp][3 + c] = hi[c];
  __syncthreads();
  if (tid < 3) {
    float l = red[0][tid], h = red[0][3 + tid];
    for (int w = 1; w < NN_WARPS; ++w) l = fminf(l, red[w][tid]), h = fmaxf(h, red[w][3 + tid]);
    ctr[blockIdx.x * 4 + tid] = 0.5f * (l + h);
  }
}

__global__ void __launch_bounds__(NN_THREADS, 2)
    nearest_kernel(const float* __restrict__ x, const float* __restrict__ y, int nx, int ny, const float* __restrict__ ctr,
                   int row_tiles, int chunks, int chunk, unsigned long long* __restrict__ keys_xy,
                   unsigned long long* __restrict__ keys_yx) {
  extern __shared__ __align__(16) float smem[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long blk = blockIdx.x;
  const int ck = (int)(blk % chunks);
  const int tile = (int)(blk / chunks % row_tiles);
  const long long pair = blk / chunks / row_tiles;
  const float* rows = x + pair * nx * 3;
  const float* cols = y + pair * ny * 3;
  const float c0x = ctr[pair * 4 + 0], c0y = ctr[pair * 4 + 1], c0z = ctr[pair * 4 + 2];
  const int col0 = ck * chunk;
  const int ncol = min(chunk, ny - col0);
  const int ncol_pad = (ncol + GROUP_COLS - 1) / GROUP_COLS * GROUP_COLS;

  float* units = smem;                                                                  // [ncol_pad / 2][8]
  unsigned long long* colkey = reinterpret_cast<unsigned long long*>(smem + ncol_pad * 4);  // [ncol_pad]
  unsigned long long* rowkey = colkey + ncol_pad;  // [ROWS_PER_TILE], entry r * 256 + tid: the row's best (value, column)

  for (int c = tid; c < ncol_pad; c += NN_THREADS) {  // pads: y = 0, |y|^2 = PAD_NORM
    float y0 = 0.f, y1 = 0.f, y2 = 0.f, n = PAD_NORM;
    if (c < ncol) {
      const long long col = col0 + c;
      y0 = __ldg(cols + col * 3 + 0) - c0x;
      y1 = __ldg(cols + col * 3 + 1) - c0y;
      y2 = __ldg(cols + col * 3 + 2) - c0z;
      n = fmaf(y2, y2, fmaf(y1, y1, y0 * y0));
    }
    // unit u of group g holds columns g*64 + u (even slot) and g*64 + 32 + u (odd slot)
    const int g = c / GROUP_COLS, r = c % GROUP_COLS, u = r & 31, hi_slot = r >> 5;
    float* t = units + (g * 32 + u) * 8 + hi_slot;
    t[0] = -2.f * y0;
    t[2] = -2.f * y1;
    t[4] = -2.f * y2;
    t[6] = n;
    colkey[c] = NO_KEY;
  }

  const int wrow0 = tile * ROWS_PER_TILE + warp * 32 * ROWS_PER_LANE;
  float2 xx[ROWS_PER_LANE], xy[ROWS_PER_LANE], xz[ROWS_PER_LANE], xn[ROWS_PER_LANE];
#pragma unroll
  for (int r = 0; r < ROWS_PER_LANE; ++r) {
    const int row = wrow0 + r * 32 + lane;
    float x0 = 0.f, x1 = 0.f, x2 = 0.f, n = PAD_NORM;
    if (row < nx) {
      x0 = __ldg(rows + (long long)row * 3 + 0) - c0x;
      x1 = __ldg(rows + (long long)row * 3 + 1) - c0y;
      x2 = __ldg(rows + (long long)row * 3 + 2) - c0z;
      n = fmaf(x2, x2, fmaf(x1, x1, x0 * x0));
    }
    xx[r] = make_float2(x0, x0);
    xy[r] = make_float2(x1, x1);
    xz[r] = make_float2(x2, x2);
    xn[r] = make_float2(n, n);
    rowkey[r * NN_THREADS + tid] = NO_KEY;
  }
  __syncthreads();

  if (wrow0 < nx) {  // warp-uniform: warps past the end of the rows skip the sweep
    uint32_t rid[ROWS_PER_LANE];  // position of each row in the warp's 256: the id of its column keys
#pragma unroll
    for (int r = 0; r < ROWS_PER_LANE; ++r) rid[r] = r * 32 + lane;
    for (int g = 0; g < ncol_pad / GROUP_COLS; ++g) {
      const float4* unit = reinterpret_cast<const float4*>(units + g * 32 * 8);
      float gk[ROWS_PER_LANE];  // row keys: minimum over the group
#pragma unroll
      for (int r = 0; r < ROWS_PER_LANE; ++r) gk[r] = INFINITY;
      float k0 = INFINITY, k1 = INFINITY;  // column keys of the unit this lane works on (even / odd slot)
#pragma unroll 4
      for (int s = 0; s < 32; ++s) {
        const uint32_t u = (lane + s) & 31, u_hi = u + 32;
        const float4 p = unit[u * 2], q = unit[u * 2 + 1];
        const float2 yx = make_float2(p.x, p.y), yy = make_float2(p.z, p.w);
        const float2 yz = make_float2(q.x, q.y), yn = make_float2(q.z, q.w);
        float ckx[ROWS_PER_LANE], cky[ROWS_PER_LANE];
#pragma unroll
        for (int r = 0; r < ROWS_PER_LANE; ++r) {
          float2 d = __fadd2_rn(xn[r], yn);
          d = __ffma2_rn(xx[r], yx, d);
          d = __ffma2_rn(xy[r], yy, d);
          d = __ffma2_rn(xz[r], yz, d);
          gk[r] = min3f(gk[r], key32<ROW_MASK>(d.x, u), key32<ROW_MASK>(d.y, u_hi));
          ckx[r] = key32<COL_MASK>(d.x, rid[r]);
          cky[r] = key32<COL_MASK>(d.y, rid[r]);
        }
#pragma unroll
        for (int r = 0; r < ROWS_PER_LANE; r += 2) {
          k0 = min3f(k0, ckx[r], ckx[r + 1]);
          k1 = min3f(k1, cky[r], cky[r + 1]);
        }
        if (s != 31) {
          k0 = __shfl_sync(0xffffffffu, k0, (lane + 1) & 31);
          k1 = __shfl_sync(0xffffffffu, k1, (lane + 1) & 31);
        }
      }
      const int u = (lane + 31) & 31;  // the unit whose keys this lane holds after the last step
      const uint32_t b0 = __float_as_uint(k0), b1 = __float_as_uint(k1);
      atomicMin(&colkey[g * GROUP_COLS + u], (unsigned long long)(b0 & COL_MASK) << 32 | (uint32_t)(wrow0 + (b0 & 0xffu)));
      atomicMin(&colkey[g * GROUP_COLS + 32 + u],
                (unsigned long long)(b1 & COL_MASK) << 32 | (uint32_t)(wrow0 + (b1 & 0xffu)));
#pragma unroll
      for (int r = 0; r < ROWS_PER_LANE; ++r) {  // this thread's own entries: no atomics
        const uint32_t b = __float_as_uint(gk[r]);
        const unsigned long long k =
            (unsigned long long)(b & ROW_MASK) << 32 | (uint32_t)(col0 + g * GROUP_COLS + (int)(b & 0x3fu));
        rowkey[r * NN_THREADS + tid] = min(rowkey[r * NN_THREADS + tid], k);
      }
    }
#pragma unroll
    for (int r = 0; r < ROWS_PER_LANE; ++r) {
      const int row = wrow0 + r * 32 + lane;
      if (row < nx) atomicMin(&keys_xy[pair * nx + row], rowkey[r * NN_THREADS + tid]);
    }
  }
  __syncthreads();
  for (int c = tid; c < ncol; c += NN_THREADS) atomicMin(&keys_yx[pair * ny + col0 + c], colkey[c]);
}

// Decodes one point's key and recomputes its distance from the caller's coordinates in difference form.
__global__ void __launch_bounds__(NN_THREADS) finish_kernel(const float* __restrict__ x, const float* __restrict__ y,
                                                            long long clouds, int nx, int ny,
                                                            const unsigned long long* __restrict__ keys,
                                                            float* __restrict__ dist_xy, int* __restrict__ idx_xy,
                                                            float* __restrict__ dist_yx, int* __restrict__ idx_yx) {
  const long long t = blockIdx.x * (long long)NN_THREADS + threadIdx.x;
  const long long nxy = clouds * nx;
  if (t >= nxy + clouds * ny) return;
  const bool fwd = t < nxy;
  const long long k = fwd ? t : t - nxy;  // point within its side
  const int n_self = fwd ? nx : ny, n_other = fwd ? ny : nx;
  const long long pair = k / n_self;
  const float* p = (fwd ? x : y) + k * 3;
  const int j = (int)(uint32_t)keys[t];
  const float* q = (fwd ? y : x) + (pair * n_other + j) * 3;
  const float d0 = __ldg(p) - __ldg(q), d1 = __ldg(p + 1) - __ldg(q + 1), d2 = __ldg(p + 2) - __ldg(q + 2);
  const float d = fmaf(d2, d2, fmaf(d1, d1, d0 * d0));
  if (fwd) {
    dist_xy[k] = d;
    idx_xy[k] = j;
  } else {
    dist_yx[k] = d;
    idx_yx[k] = j;
  }
}

long long keys_words(long long clouds, int nx, int ny) { return clouds * ((long long)nx + ny); }

}  // namespace
}  // namespace gecco

extern "C" int64_t gecco_nearest_scratch_bytes(int32_t clouds, int32_t nx, int32_t ny) {
  if (clouds < 0 || nx < 0 || ny < 0) return -1;
  return (int64_t)(gecco::keys_words(clouds, nx, ny) + 2LL * clouds) * 8;  // keys, then a float4 centre per pair
}

extern "C" int gecco_nearest(const gecco_nearest_args* args, void* stream) {
  using namespace gecco;
  GECCO_REQUIRE(args != nullptr, "nearest: null args");
  const gecco_nearest_args& A = *args;
  GECCO_REQUIRE(A.clouds >= 0, "nearest: negative cloud count");
  GECCO_REQUIRE(A.nx >= 1 && A.ny >= 1 && A.nx <= MAX_POINTS && A.ny <= MAX_POINTS,
                "nearest: clouds need 1 to %d points (got %d and %d)", MAX_POINTS, A.nx, A.ny);
  if (A.clouds == 0) return GECCO_OK;  // (empty tensors may have null data pointers)
  GECCO_REQUIRE(A.x && A.y && A.dist_xy && A.idx_xy && A.dist_yx && A.idx_yx && A.scratch, "nearest: null argument");
  const int64_t need = gecco_nearest_scratch_bytes(A.clouds, A.nx, A.ny);
  GECCO_REQUIRE(A.scratch_bytes >= need, "nearest: scratch of %lld bytes, need %lld", (long long)A.scratch_bytes,
                (long long)need);
  GECCO_REQUIRE(((uintptr_t)A.scratch & 15) == 0, "nearest: scratch must be 16-byte aligned");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const long long words = keys_words(A.clouds, A.nx, A.ny);
  auto* keys = static_cast<unsigned long long*>(A.scratch);
  float* ctr = reinterpret_cast<float*>(keys + words);

  // columns per block: the largest power of two (2048 down to 128) that still gives 8 blocks per SM
  int dev = 0, sms = 148;
  cudaError_t e = cudaGetDevice(&dev);
  if (e == cudaSuccess) e = cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  if (e != cudaSuccess) return fail_cuda(e, "nearest: device attribute");
  const int row_tiles = (A.nx + ROWS_PER_TILE - 1) / ROWS_PER_TILE;
  int chunk = MAX_CHUNK;
  auto chunks_of = [&](int c) { return (A.ny + c - 1) / c; };
  while (chunk > MIN_CHUNK && (long long)A.clouds * row_tiles * chunks_of(chunk) < 8LL * sms) chunk /= 2;
  const int chunks = chunks_of(chunk);
  const long long blocks = (long long)A.clouds * row_tiles * chunks;
  GECCO_REQUIRE(blocks <= 0x7fffffffLL, "nearest: too many blocks (%lld)", blocks);
  const long long finish_blocks = (words + NN_THREADS - 1) / NN_THREADS;
  GECCO_REQUIRE(finish_blocks <= 0x7fffffffLL, "nearest: too many points (%lld)", words);

  e = cudaMemsetAsync(keys, 0xff, (size_t)words * 8, s);
  if (e != cudaSuccess) return fail_cuda(e, "nearest: key initialisation");
  centre_kernel<<<(unsigned)A.clouds, NN_THREADS, 0, s>>>(A.x, A.nx, ctr);
  GECCO_CHECK_LAUNCH("nearest centre_kernel");
  const size_t smem = (size_t)chunk * 24 + (size_t)ROWS_PER_TILE * 8;
  if (smem > 48 * 1024) {  // host-side attribute, no synchronisation
    e = cudaFuncSetAttribute(nearest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return fail_cuda(e, "nearest: shared memory attribute");
  }
  nearest_kernel<<<(unsigned)blocks, NN_THREADS, smem, s>>>(A.x, A.y, A.nx, A.ny, ctr, row_tiles, chunks, chunk, keys,
                                                            keys + (long long)A.clouds * A.nx);
  GECCO_CHECK_LAUNCH("nearest_kernel");
  finish_kernel<<<(unsigned)finish_blocks, NN_THREADS, 0, s>>>(A.x, A.y, A.clouds, A.nx, A.ny, keys, A.dist_xy, A.idx_xy,
                                                               A.dist_yx, A.idx_yx);
  GECCO_CHECK_LAUNCH("nearest finish_kernel");
  return GECCO_OK;
}
