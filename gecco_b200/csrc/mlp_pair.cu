// Point-side MLP of a BroadcastingLayer (models/set_transformer.py:165-166, models/mlp.py:5-39, activation.py:17-24)
//     x <- x + W2 . g(W1 . AdaGN(x) + b1) + b2
// as ONE persistent CTA-pair tcgen05 kernel in which the 768-wide hidden activation never reaches HBM.
//
// Per 256-row block a CTA pair runs six 256 x 192 tiles through the same two TMEM accumulator slots:
//     U0..U3 : hidden columns [192 j, 192 j + 192) = g(A' W1_j^T + b1),  A' = AdaGN(xb) normalised in place in the resident
//              A tile exactly as in gemm_pair.cu (kANorm); the fast bf16 epilogue writes the tile into a per-CTA SCRATCH
//              [128 rows x 768] in global memory -- 28 MB for the whole grid, rewritten every row block, so it lives in L2;
//     D0, D1 : output columns [192 j, ..) = H W2_j^T + b2 + x, K = 768: the hidden k-blocks come back from the scratch by
//              TMA through the SIX SLOTS OF THE A TILE (free during this phase), the weights through the same ring as W1.
// The epilogue of D1 runs under U0 / U1 of the next row block.  Compared with the two GEMMs of rounds 1-2 the hidden
// tensor costs no HBM traffic (402 MB per layer at 64 x 2048 points) and one launch disappears.
//
// The residual epilogue cannot afford the 64 KB of TMA-fed X buffers of epilogue.cuh next to a resident A tile and a weight
// ring, so here every epilogue WARP owns one 4 KB staging block: the fp32 residual chunk of its 32 rows is fetched with
// coalesced LDG.128 one chunk ahead (registers are the prefetch buffer; the producer warp pulls each output tile's
// residual into L2 with TMA prefetches in the D phase, so the loads hit L2), written into the block, read back row-per-thread, and
// the finished rows leave through the same block by one bulk tensor store.  No loader warp, no cross-warp barrier.
//
//   warp 0 : TMA producer            warps 2-3 : A-operand transform (AdaGN)
//   warp 1 : MMA issuer (leader)     warps 4-11: epilogue
#include "common.cuh"
#include "debug_api.h"
#include "epilogue.cuh"
#include "kernels.cuh"
#include "norm.cuh"
#include "ptx.cuh"

namespace gecco {
extern long long* g_gemm_debug;
namespace {

constexpr int BM = 128;
constexpr int BN = 192;
constexpr int BNH = BN / 2;
constexpr int BK = 64;
constexpr int C = 384;
constexpr int HID = 768;
constexpr int KB1 = C / BK;      // 6  k-blocks of the first product = slots of the A tile
constexpr int KB2 = HID / BK;    // 12 k-blocks of the second product
constexpr int NU = HID / BN;     // 4  tiles of the first product per row block
constexpr int ND = C / BN;       // 2  tiles of the second product
constexpr int A_KB_BYTES = BM * BK * 2;      // 16 KiB
constexpr int B_STAGE_BYTES = BNH * BK * 2;  // 12 KiB
constexpr int BST = 6;                       // weight ring depth
constexpr int ACC_COLS = 256;
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 128 + EPI_GROUPS * EPI_THREADS;
constexpr int XF_THREADS = 64;
constexpr int NORM_BYTES = 2 * 2 * C * 4;     // a[K], s[K], double buffered over row blocks
constexpr int X_BYTES = 8 * 4096;             // per-warp fp32 staging blocks (32 rows x 128 B, SWIZZLE_128B)
constexpr int O16_BYTES = 8 * 2048;           // per-warp bf16 staging blocks (32 rows x 64 B, SWIZZLE_64B)
constexpr int SMEM_BYTES = 1024 + KB1 * A_KB_BYTES + NORM_BYTES + BST * B_STAGE_BYTES + X_BYTES + O16_BYTES + EPI_BIAS_BYTES + 512;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct MParams {
  EpiParams u;   // first product: bias b1, activation
  EpiParams d;   // second product: bias b2, residual, statistics, fp32 / bf16 outputs
  const float* res; long long ldr;
  int num_pair_blocks;
  // A-operand normalisation
  const double* n_stats; int n_stat_gs, n_groups; float n_eps;
  const float* n_t; int n_t_stride;
  const float *n_scale_w, *n_scale_b, *n_bias_w, *n_bias_b;
  long long* dbg;
};

// L2 residency policies (ptx.cuh l2_policy kinds): the A operand and the residual are read once (evict_first), the hidden
// tiles parked in the scratch are read back by the second product (evict_last), the outputs get the default
constexpr int POL_A = 1, POL_RES = 1, POL_HIDDEN = 2, POL_OUT = 0;

// physical row block of the pb-th one: row blocks are walked from the end, so the previous kernel's last writes are read
// first, while still in L2
#define RB(pb) (p.num_pair_blocks - 1 - (pb))
// development aid: cycles spent in a barrier wait, accumulated when the debug buffer is set (gecco_set_debug_buffer)
#define TW(acc, bar, parity)              \
  do {                                    \
    if (p.dbg != nullptr) {               \
      const long long t0__ = clock64();   \
      mbar_wait(bar, parity);             \
      acc += clock64() - t0__;            \
    } else {                              \
      mbar_wait(bar, parity);             \
    }                                     \
  } while (0)

// Waits until all bulk stores of this thread have COMPLETED (their global writes are visible), not only read their source.
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ float4 ldg128(const float* p, uint64_t pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0,%1,%2,%3}, [%4], %5;" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p), "l"(pol));
  return v;
}

// The fp32 residual chunk (32 rows x 32 columns) of a warp, one 16-byte piece of four rows per lane and instruction.
struct ResRegs { float4 r[8]; };
__device__ __forceinline__ void res_load(const MParams& p, int row0, int col0, int lane, ResRegs& R) {
  const float* base = p.res + (long long)(row0 + (lane >> 3)) * p.ldr + col0 + (lane & 7) * 4;
  const uint64_t pol = l2_policy(POL_RES);
#pragma unroll
  for (int i = 0; i < 8; ++i) R.r[i] = ldg128(base + (long long)(4 * i) * p.ldr, pol);
}
__device__ __forceinline__ void res_stage(uint32_t xs, int lane, const ResRegs& R) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const uint32_t row = 4 * i + (lane >> 3), piece = lane & 7;
    sts128(xs + row * 128u + ((piece ^ (row & 7u)) << 4), R.r[i].x, R.r[i].y, R.r[i].z, R.r[i].w);
  }
}

// One 128 x 192 panel of the second product for this warp's 32 rows: chunks grp, grp + 2, grp + 4.  `R` holds the residual
// of the first chunk on entry and of the NEXT panel's first chunk (next_row0 / next_col0, or nothing when next_row0 < 0)
// on exit.
template <bool kStats>
__device__ __forceinline__ void epi_panel_ldg(const MParams& p, const EpiThread& t, const CUtensorMap* tma_o32,
                                              const CUtensorMap* tma_o16, uint32_t taddr, int m0, int n0, ResRegs& R,
                                              int next_row0, int next_col0) {
  const EpiParams& e = p.d;
  const int row0 = m0 + t.q * 32;
  const int cloud = row0 / e.rows_per_cloud;
  const int row_in_cloud = row0 + t.lane - cloud * e.rows_per_cloud;
  const bool row_valid = row_in_cloud < e.valid_rows;
  const bool rows_valid = (row0 + 31 - cloud * e.rows_per_cloud) < e.valid_rows;
  uint32_t rr[2][EPI_CHUNK];
  const uint32_t ta = taddr + t.grp * EPI_CHUNK;
  tmem_ld32_issue(ta, rr[0]);
  float st[kStats ? 32 : 1];
#pragma unroll
  for (int i = 0; i < (kStats ? 32 : 1); ++i) st[i] = 0.f;
  const uint32_t xw = t.xw0, xs = t.xs0;

  auto step = [&](auto kc) {
    constexpr int k = decltype(kc)::value;
    const int col0 = n0 + (2 * k + t.grp) * EPI_CHUNK;
    float4 b[EPI_CHUNK / 4];
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) b[j] = lds128(t.bias + k * 128u + j * 16u);
    // the previous chunk's bulk stores have read the staging blocks: the residual chunk goes in
    if (t.lane == 0) tma_store_wait_read<0>();
    __syncwarp();
    res_stage(xs, t.lane, R);
    // the following chunk's residual is in flight while this one is processed
    if (k < 2) res_load(p, row0, n0 + (2 * k + 2 + t.grp) * EPI_CHUNK, t.lane, R);
    else if (next_row0 >= 0) res_load(p, next_row0, next_col0, t.lane, R);
    __syncwarp();
    tmem_ld32_wait(rr[k & 1]);
    float v[EPI_CHUNK];
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) {
      v[4 * j + 0] = __uint_as_float(rr[k & 1][4 * j + 0]) + b[j].x;
      v[4 * j + 1] = __uint_as_float(rr[k & 1][4 * j + 1]) + b[j].y;
      v[4 * j + 2] = __uint_as_float(rr[k & 1][4 * j + 2]) + b[j].z;
      v[4 * j + 3] = __uint_as_float(rr[k & 1][4 * j + 3]) + b[j].w;
    }
    if (k < 2) tmem_ld32_issue(ta + (2 * k + 2) * EPI_CHUNK, rr[(k + 1) & 1]);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float4 x[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] = lds128(xw | (((4 * h + j) << 4) ^ t.x7));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[16 * h + 4 * j + 0] += x[j].x; v[16 * h + 4 * j + 1] += x[j].y;
        v[16 * h + 4 * j + 2] += x[j].z; v[16 * h + 4 * j + 3] += x[j].w;
      }
    }
    if (!rows_valid && !row_valid) {
#pragma unroll
      for (int j = 0; j < EPI_CHUNK; ++j) v[j] = 0.f;  // padding rows stay exactly zero
    }
    if (kStats) {
#pragma unroll
      for (int j = 0; j < EPI_CHUNK; ++j) {
        // chunk index inside the panel is 2 k + grp: instantiate both, select at run time (grp is warp-uniform)
        const int g0 = ((2 * k) * EPI_CHUNK + j) / 12, g1 = ((2 * k + 1) * EPI_CHUNK + j) / 12;
        if (t.grp == 0) {
          st[2 * g0] += v[j];
          st[2 * g0 + 1] = fmaf(v[j], v[j], st[2 * g0 + 1]);
        } else {
          st[2 * g1] += v[j];
          st[2 * g1 + 1] = fmaf(v[j], v[j], st[2 * g1 + 1]);
        }
      }
    }
    __syncwarp();  // every lane has read its residual row before the rows are overwritten (rows are thread-private, but
                   // the residual pieces were written by other lanes: keep the block coherent per phase)
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) sts128(xw | ((j << 4) ^ t.x7), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 8; ++j)
      sts128u(t.w16 | ((j << 4) ^ t.x3), pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
              pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
    fence_proxy_async_smem();
    __syncwarp();
    if (elect_one()) {
      tma_store_2d_addr_h(tma_o32, xs, col0, row0, l2_policy(POL_OUT));
      tma_store_2d_addr_h(tma_o16, t.s16, col0, row0, l2_policy(POL_OUT));
      tma_store_commit();
    }
  };
  step(std::integral_constant<int, 0>{});
  step(std::integral_constant<int, 1>{});
  step(std::integral_constant<int, 2>{});
  if constexpr (kStats) {
    const float mine = warp_reduce_scatter32(st, t.lane);
    const int gidx = (n0 / 12) * 2 + t.lane;  // [group][{sum, sumsq}]
    atomicAdd(e.stats + (long long)cloud * (e.n_out / 12) * 2 + gidx, static_cast<double>(mine));
  }
}

template <bool kStats>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
mlp_pair_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w1,
                const __grid_constant__ CUtensorMap tma_w2, const __grid_constant__ CUtensorMap tma_hs,
                const __grid_constant__ CUtensorMap tma_hl, const __grid_constant__ CUtensorMap tma_res,
                const __grid_constant__ CUtensorMap tma_o32, const __grid_constant__ CUtensorMap tma_o16, const MParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                                     // [KB1] A k-blocks | hidden k-blocks (D phase)
  float* sNorm = reinterpret_cast<float*>(smem + KB1 * A_KB_BYTES);
  uint8_t* sB = smem + KB1 * A_KB_BYTES + NORM_BYTES;                     // [BST] weight half tiles
  EpiSmem es;
  es.x0 = sB + BST * B_STAGE_BYTES;                                       // [8 warps] x 4 KB
  es.x1 = es.x0;
  es.o16 = es.x0 + X_BYTES;                                               // [8 warps] x 2 KB
  es.bias = es.o16 + O16_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(es.bias + EPI_BIAS_BYTES);
  uint64_t* a_full = bars;                 // [KB1] leader: transformed A k-block of both CTAs
  uint64_t* a_landed = a_full + KB1;       // [KB1] each CTA: raw A k-block landed
  uint64_t* h_full = a_landed + KB1;       // [KB1] leader: hidden k-block of both CTAs landed
  uint64_t* a_empty = h_full + KB1;        // [KB1] each CTA: slot consumed
  uint64_t* b_full = a_empty + KB1;        // [BST] leader
  uint64_t* b_empty = b_full + BST;        // [BST] each CTA
  uint64_t* acc_full = b_empty + BST;      // [2] each CTA
  uint64_t* acc_empty = acc_full + 2;      // [2] leader
  uint64_t* h_ready = acc_empty + 2;       // [NU] each CTA: hidden tile j of this CTA's rows is in the scratch
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(h_ready + NU);
  es.res_full = es.res_empty = nullptr;

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const uint32_t urank = uniform_u32(rank);
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int srow = blockIdx.x * BM;  // this CTA's rows in the hidden scratch

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a); tma_prefetch_desc(&tma_w1); tma_prefetch_desc(&tma_w2); tma_prefetch_desc(&tma_hs);
    tma_prefetch_desc(&tma_hl); tma_prefetch_desc(&tma_res); tma_prefetch_desc(&tma_o32); tma_prefetch_desc(&tma_o16);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < KB1; ++i) {
      mbar_init(&a_full[i], 2 * (XF_THREADS / 32));
      mbar_init(&a_landed[i], 1);
      mbar_init(&h_full[i], 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < BST; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 2 * EPI_GROUPS * EPI_THREADS / 32);
    }
    for (int i = 0; i < NU; ++i) mbar_init(&h_ready[i], EPI_GROUPS * EPI_THREADS / 32);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair<TMEM_COLS>(tmem_slot);
  tc_fence_before_sync();
  cluster_sync_all();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch_dependents();

  if (warp < 4) {
    setmaxnreg_dec<104>();
    if (warp == 0 && lane == 0) {
      // ------------------------------------------------------------ TMA producer (both CTAs)
      int stage = 0;
      uint32_t bphase = 0;
      uint32_t it = 0;
      long long w_b1 = 0, w_a = 0, w_hr = 0, w_hs = 0, w_b2 = 0;
      const long long t_start = clock64();
      const uint64_t h_pol = l2_policy(POL_HIDDEN);  // hidden k-blocks coming back from the scratch
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
        const int m0 = RB(pb) * 2 * BM + (int)rank * BM;
        // first product: A k-blocks once per row block, W1 half tiles per (tile, k-block)
        for (int nb = 0; nb < NU; ++nb) {
          const int wrow = nb * BN + (int)rank * BNH;
          for (int kb = 0; kb < KB1; ++kb) {
            TW(w_b1, &b_empty[stage], bphase ^ 1u);
            if (rank == 0) mbar_arrive_expect_tx(&b_full[stage], 2 * B_STAGE_BYTES);
            if (nb == 0) {
              TW(w_a, &a_empty[kb], ((it * 5u) & 1u) ^ 1u);  // fill 5 it of the slot
              mbar_arrive_expect_tx(&a_landed[kb], A_KB_BYTES);
              tma_load_2d_h(sA + kb * A_KB_BYTES, &tma_a, &a_landed[kb], kb * BK, m0, l2_policy(POL_A));
            }
            tma_load_2d_pair(sB + stage * B_STAGE_BYTES, &tma_w1, &b_full[stage], kb * BK, wrow);
            if (++stage == BST) { stage = 0; bphase ^= 1u; }
          }
        }
        // the A tile of the next row block -> L2
        if (pb + num_pairs < p.num_pair_blocks)
          for (int kb = 0; kb < KB1; ++kb) tma_prefetch_l2_2d(&tma_a, kb * BK, RB(pb + num_pairs) * 2 * BM + (int)rank * BM);
        // second product: hidden k-blocks from the scratch through the slots of the A tile, W2 half tiles
        for (int nb = 0; nb < ND; ++nb) {
          const int wrow = nb * BN + (int)rank * BNH;
          // the residual of this output tile -> L2
          for (int c = 0; c < BN / EPI_CHUNK; ++c) tma_prefetch_l2_2d(&tma_res, nb * BN + c * EPI_CHUNK, m0);
          for (int kb = 0; kb < KB2; ++kb) {
            const int slot = kb % KB1;
            const uint32_t fill = it * 5u + 1u + (uint32_t)(nb * 2 + kb / KB1);
            if (nb == 0 && kb % (BN / BK) == 0) TW(w_hr, &h_ready[kb / (BN / BK)], it & 1u);
            TW(w_hs, &a_empty[slot], (fill & 1u) ^ 1u);
            if (rank == 0) mbar_arrive_expect_tx(&h_full[slot], 2 * A_KB_BYTES);
            tma_load_2d_pair_h(sA + slot * A_KB_BYTES, &tma_hl, &h_full[slot], kb * BK, srow, h_pol);
            TW(w_b2, &b_empty[stage], bphase ^ 1u);
            if (rank == 0) mbar_arrive_expect_tx(&b_full[stage], 2 * B_STAGE_BYTES);
            tma_load_2d_pair(sB + stage * B_STAGE_BYTES, &tma_w2, &b_full[stage], kb * BK, wrow);
            if (++stage == BST) { stage = 0; bphase ^= 1u; }
          }
        }
      }
      if (p.dbg != nullptr) {
        long long* d = p.dbg + (long long)blockIdx.x * 32;
        d[0] = clock64() - t_start; d[1] = w_b1; d[2] = w_a; d[3] = w_hr; d[4] = w_hs; d[5] = w_b2;
      }
    } else if (uwarp == 1) {
      // ------------------------------------------------------------ MMA issuer (leader CTA)
      if (urank == 0) {
        constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN);
        const uint32_t sA_u = uniform_u32(smem_u32(sA)), sB_u = uniform_u32(smem_u32(sB));
        const uint32_t tmem_u = uniform_u32(tmem_base);
        int stage = 0;
        uint32_t bphase = 0;
        uint32_t it = 0, tile = 0;
        long long m_accu = 0, m_b1 = 0, m_a = 0, m_accd = 0, m_h = 0, m_b2 = 0;
        const long long t_start = clock64();
        for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
          for (int nb = 0; nb < NU; ++nb, ++tile) {
            const uint32_t slot = tile & 1u;
            TW(m_accu, &acc_empty[slot], ((tile >> 1) & 1u) ^ 1u);
            tc_fence_after_sync();
            const uint32_t tmem_d = tmem_u + slot * ACC_COLS;
            for (int kb = 0; kb < KB1; ++kb) {
              TW(m_b1, &b_full[stage], bphase);
              if (nb == 0) TW(m_a, &a_full[kb], it & 1u);
              tc_fence_after_sync();
              const uint64_t da = umma_desc_k_sw128(sA_u + kb * A_KB_BYTES);
              const uint64_t db = umma_desc_k_sw128(sB_u + stage * B_STAGE_BYTES);
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_bf16_ss_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                umma_commit_pair(&b_empty[stage]);
                if (nb == NU - 1) umma_commit_pair(&a_empty[kb]);  // the slot goes to the hidden k-blocks
              }
              __syncwarp();
              if (++stage == BST) { stage = 0; bphase ^= 1u; }
            }
            if (elect_one()) umma_commit_pair(&acc_full[slot]);
            __syncwarp();
          }
          for (int nb = 0; nb < ND; ++nb, ++tile) {
            const uint32_t slot = tile & 1u;
            TW(m_accd, &acc_empty[slot], ((tile >> 1) & 1u) ^ 1u);
            tc_fence_after_sync();
            const uint32_t tmem_d = tmem_u + slot * ACC_COLS;
            for (int kb = 0; kb < KB2; ++kb) {
              const int as = kb % KB1;
              const uint32_t hfill = it * 4u + (uint32_t)(nb * 2 + kb / KB1);
              TW(m_h, &h_full[as], hfill & 1u);
              TW(m_b2, &b_full[stage], bphase);
              tc_fence_after_sync();
              const uint64_t da = umma_desc_k_sw128(sA_u + as * A_KB_BYTES);
              const uint64_t db = umma_desc_k_sw128(sB_u + stage * B_STAGE_BYTES);
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_bf16_ss_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                umma_commit_pair(&b_empty[stage]);
                umma_commit_pair(&a_empty[as]);
              }
              __syncwarp();
              if (++stage == BST) { stage = 0; bphase ^= 1u; }
            }
            if (elect_one()) umma_commit_pair(&acc_full[slot]);
            __syncwarp();
          }
        }
        if (p.dbg != nullptr && lane == 0) {
          long long* d = p.dbg + (long long)blockIdx.x * 32;
          d[6] = clock64() - t_start; d[7] = m_accu; d[8] = m_b1; d[9] = m_a; d[10] = m_accd; d[11] = m_h; d[12] = m_b2;
        }
      }
    } else if (uwarp == 2 || uwarp == 3) {
      // ------------------------------------------------------------ A-operand transform (see gemm_pair.cu)
      const int tt = threadIdx.x - 64;
      const uint32_t pj = (uint32_t)tt & 7u, rl = (uint32_t)tt >> 3;
      const uint32_t lj = pj ^ rl;
      const int gs = C / p.n_groups;
      const double inv_count = 1.0 / ((double)p.d.valid_rows * gs);
      auto make_norm = [&](int pb, uint32_t buf) {
        const int m0 = RB(pb) * 2 * BM + (int)rank * BM;
        const int cloud = m0 / p.d.rows_per_cloud;
        const double* cst = p.n_stats + (long long)cloud * (C / p.n_stat_gs) * 2;
        float* na = sNorm + buf * 2 * C;
        float* ns = na + C;
        const float tc = __ldg(p.n_t + (long long)cloud * p.n_t_stride);
        const int per = gs / p.n_stat_gs;
        constexpr int NCH = C / XF_THREADS;
        double s1[NCH], s2[NCH];
        float sw[NCH], sb[NCH], bw[NCH], bb[NCH];
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int c = tt + i * XF_THREADS;
          const int g = c / gs;
          s1[i] = s2[i] = 0.0;
          for (int j = 0; j < per; ++j) {
            s1[i] += cst[(g * per + j) * 2];
            s2[i] += cst[(g * per + j) * 2 + 1];
          }
          sw[i] = __ldg(p.n_scale_w + c); sb[i] = __ldg(p.n_scale_b + c);
          bw[i] = __ldg(p.n_bias_w + c); bb[i] = __ldg(p.n_bias_b + c);
        }
#pragma unroll
        for (int i = 0; i < NCH; ++i) {
          const int c = tt + i * XF_THREADS;
          const double m = s1[i] * inv_count;
          double var = fma(-m, m, s2[i] * inv_count);
          if (var < 0.0) var = 0.0;
          const float rstd = rsqrtf(static_cast<float>(var) + p.n_eps);
          const float a = (tc * sw[i] + sb[i]) * rstd;
          na[c] = a;
          ns[c] = (tc * bw[i] + bb[i]) - a * static_cast<float>(m);
        }
        named_bar_sync(2, XF_THREADS);
      };
      uint32_t it = 0;
      const uint32_t row0 = smem_u32(sA) + rl * 128u + (pj << 4);
      if (pair < p.num_pair_blocks) make_norm(pair, 0);
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
        const uint32_t na_u = smem_u32(sNorm + (it & 1u) * 2 * C), ns_u = na_u + C * 4;
        for (int kb = 0; kb < KB1; ++kb) {
          const uint32_t ko = (uint32_t)(kb * BK) * 4u + lj * 32u;
          const float4 a0 = lds128(na_u + ko), a1 = lds128(na_u + ko + 16u);
          const float4 s0 = lds128(ns_u + ko), s1 = lds128(ns_u + ko + 16u);
          mbar_wait(&a_landed[kb], it & 1u);
          const uint32_t base = row0 + kb * A_KB_BYTES;
#pragma unroll
          for (int b = 0; b < 2; ++b) {
            uint4 v[8];
#pragma unroll
            for (int i = 0; i < 8; ++i)
              asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(v[i].x), "=r"(v[i].y), "=r"(v[i].z), "=r"(v[i].w)
                           : "r"(base + (uint32_t)(8 * b + i) * 1024u));
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const float x0 = __uint_as_float(v[i].x << 16), x1 = __uint_as_float(v[i].x & 0xffff0000u);
              const float x2 = __uint_as_float(v[i].y << 16), x3 = __uint_as_float(v[i].y & 0xffff0000u);
              const float x4 = __uint_as_float(v[i].z << 16), x5 = __uint_as_float(v[i].z & 0xffff0000u);
              const float x6 = __uint_as_float(v[i].w << 16), x7 = __uint_as_float(v[i].w & 0xffff0000u);
              sts128u(base + (uint32_t)(8 * b + i) * 1024u,
                      pack_bf16x2(fmaf(a0.x, x0, s0.x), fmaf(a0.y, x1, s0.y)), pack_bf16x2(fmaf(a0.z, x2, s0.z), fmaf(a0.w, x3, s0.w)),
                      pack_bf16x2(fmaf(a1.x, x4, s1.x), fmaf(a1.y, x5, s1.y)), pack_bf16x2(fmaf(a1.z, x6, s1.z), fmaf(a1.w, x7, s1.w)));
            }
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) mbar_arrive_leader(&a_full[kb]);
        }
        if (pb + num_pairs < p.num_pair_blocks) make_norm(pb + num_pairs, (it & 1u) ^ 1u);
      }
    }
  } else {
    setmaxnreg_inc<200>();
    // ------------------------------------------------------------ epilogue (each CTA: its own 128 rows)
    const EpiThread et = epi_thread_init(es, (warp - 4) >> 2, threadIdx.x & (EPI_THREADS - 1));
    const int q = warp & 3;
    uint32_t tile = 0, it = 0;
    EpiBias bias_r;
    ResRegs R;
    long long e_accu = 0, e_fast = 0, e_store = 0, e_accd = 0, e_panel = 0;
    const long long e_start = clock64();
    if (pair < p.num_pair_blocks) epi_bias_load(p.u, et, RB(pair) * 2 * BM + (int)rank * BM, 0, bias_r);
    for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
      const int m0 = RB(pb) * 2 * BM + (int)rank * BM;
      const bool row_valid = (m0 % p.u.rows_per_cloud) + q * 32 + (int)et.lane < p.u.valid_rows;
      for (int nb = 0; nb < NU; ++nb, ++tile) {
        const uint32_t slot = tile & 1u;
        epi_bias_stage(p.u, et, bias_r);
        if (nb + 1 < NU) epi_bias_load(p.u, et, m0, (nb + 1) * BN, bias_r);
        else epi_bias_load(p.d, et, m0, 0, bias_r);
        TW(e_accu, &acc_full[slot], (tile >> 1) & 1u);
        tc_fence_after_sync();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot * ACC_COLS;
        long long tf0 = 0, tf1 = 0;
        if (p.dbg != nullptr) tf0 = clock64();
        epi_tile_fast<true>(p.u, et, &tma_hs, taddr, srow, nb * BN, smem_u32(es.o16), row_valid, [&] {
          tc_fence_before_sync();
          __syncwarp();
          if (et.lane == 0) mbar_arrive_leader(&acc_empty[slot]);
        });
        if (p.dbg != nullptr) tf1 = clock64();
        // the tile's hidden columns of this warp's rows are in the scratch (L2): the producer may load them back
        if (et.lane == 0) {
          tma_store_wait_all();
          mbar_arrive(&h_ready[nb]);
        }
        __syncwarp();
        if (p.dbg != nullptr) { e_fast += tf1 - tf0; e_store += clock64() - tf1; }
        if (nb == NU - 1) res_load(p, m0 + q * 32, et.grp * EPI_CHUNK, et.lane, R);  // residual of the first D chunk
      }
      for (int nb = 0; nb < ND; ++nb, ++tile) {
        const uint32_t slot = tile & 1u;
        epi_bias_stage(p.d, et, bias_r);
        if (nb + 1 < ND) epi_bias_load(p.d, et, m0, (nb + 1) * BN, bias_r);
        else if (pb + num_pairs < p.num_pair_blocks) epi_bias_load(p.u, et, RB(pb + num_pairs) * 2 * BM + (int)rank * BM, 0, bias_r);
        TW(e_accd, &acc_full[slot], (tile >> 1) & 1u);
        tc_fence_after_sync();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot * ACC_COLS;
        long long tp0 = 0;
        if (p.dbg != nullptr) tp0 = clock64();
        epi_panel_ldg<kStats>(p, et, &tma_o32, &tma_o16, taddr, m0, nb * BN, R, nb + 1 < ND ? m0 + q * 32 : -1,
                              (nb + 1) * BN + et.grp * EPI_CHUNK);
        if (p.dbg != nullptr) e_panel += clock64() - tp0;
        tc_fence_before_sync();
        __syncwarp();
        if (et.lane == 0) mbar_arrive_leader(&acc_empty[slot]);
      }
    }
    if (et.lane == 0) tma_store_wait_read<0>();
    if (p.dbg != nullptr && threadIdx.x == 128) {
      long long* d = p.dbg + (long long)blockIdx.x * 32;
      d[13] = clock64() - e_start; d[14] = e_accu; d[15] = e_fast; d[16] = e_store; d[17] = e_accd; d[18] = e_panel;
    }
  }

  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc_pair<TMEM_COLS>(tmem_base);
  }
}

}  // namespace

bool mlp_pair_supported(const gecco_mlp_args& a) {
  return a.anorm.stats != nullptr && a.c == C && a.hidden == HID && a.m > 0 && a.m % (2 * BM) == 0 &&
         a.rows_per_cloud % (2 * BM) == 0 && a.w1_rows_per_cloud == 0 && a.scratch != nullptr && a.res != nullptr &&
         a.out_f32 != nullptr && a.out_bf16 != nullptr && a.anorm.groups > 0 && a.anorm.groups <= 128 && C % a.anorm.groups == 0 &&
         a.anorm.stat_gs > 0 && (C / a.anorm.groups) % a.anorm.stat_gs == 0 && sm_count() >= 2 && g_use_pairs_ref();
}

int launch_mlp_pair(const gecco_mlp_args& a, cudaStream_t stream) {
  GECCO_REQUIRE(mlp_pair_supported(a), "mlp (pair kernel): unsupported shape or missing A-operand normalisation / scratch");
  GECCO_REQUIRE(a.a && a.w1 && a.w2 && a.b1 && a.b2, "mlp: null operand");
  GECCO_REQUIRE(a.valid_rows > 0 && a.valid_rows <= a.rows_per_cloud, "mlp: valid_rows out of range");
  GECCO_REQUIRE(a.act_alpha != 0.f, "mlp: act_alpha must be non-zero");
  GECCO_REQUIRE(a.anorm.t && a.anorm.scale_w && a.anorm.scale_b && a.anorm.bias_w && a.anorm.bias_b, "mlp: incomplete AdaGN");

  const int num_pair_blocks = a.m / (2 * BM);
  int pairs = sm_count() / 2;
  if (pairs > num_pair_blocks) pairs = num_pair_blocks;
  const int grid = 2 * pairs;

  CUtensorMap ta, tw1, tw2, ths, thl, tres, t32, t16;
  if (int rc = make_tmap_bf16(&ta, a.a, C, a.m, a.lda, BM)) return rc;
  if (int rc = make_tmap_bf16(&tw1, a.w1, C, HID, a.ldw1, BNH)) return rc;
  if (int rc = make_tmap_bf16(&tw2, a.w2, HID, C, a.ldw2, BNH)) return rc;
  if (int rc = make_tmap(&ths, 2, a.scratch, HID, (uint64_t)grid * BM, HID * 2, EPI_CHUNK, 32, 64)) return rc;
  if (int rc = make_tmap_bf16(&thl, a.scratch, HID, (uint64_t)grid * BM, HID, BM)) return rc;
  if (int rc = make_residual_tmap(a.res, a.ldr, a.m, C, ta, &tres)) return rc;
  if (int rc = make_output_tmaps(a.out_f32, a.ldo32, a.out_bf16, a.ldo16, a.m, C, ta, &t32, &t16)) return rc;

  MParams p = {};
  auto base = [&](EpiParams& e, int n_out) {
    e.M = a.m; e.n_out = n_out;
    e.rows_per_cloud = a.rows_per_cloud; e.valid_rows = a.valid_rows;
    e.bias_stride = 0; e.act = 0; e.act_k = 0.f; e.has_res = 0;
    e.o32 = nullptr; e.o16 = nullptr; e.stats = nullptr;
    e.geom = nullptr; e.sigma = nullptr; e.sigma_stride = 0; e.sigma_data = 1.f; e.wx = nullptr;
    e.skip = 0; e.dbg = nullptr;
  };
  base(p.u, HID);
  p.u.bias = a.b1; p.u.act = 1;
  p.u.act_k = static_cast<float>(-1.4426950408889634 / (2.0 * (double)a.act_alpha * (double)a.act_alpha));
  p.u.o16 = static_cast<__nv_bfloat16*>(a.scratch);
  base(p.d, C);
  p.d.bias = a.b2; p.d.has_res = 1; p.d.o32 = a.out_f32; p.d.o16 = static_cast<__nv_bfloat16*>(a.out_bf16);
  p.d.stats = a.stats;
  p.res = a.res; p.ldr = a.ldr;
  p.num_pair_blocks = num_pair_blocks;
  p.n_stats = a.anorm.stats; p.n_stat_gs = a.anorm.stat_gs; p.n_groups = a.anorm.groups; p.n_eps = a.anorm.eps;
  p.n_t = a.anorm.t; p.n_t_stride = a.anorm.t_stride;
  p.n_scale_w = a.anorm.scale_w; p.n_scale_b = a.anorm.scale_b; p.n_bias_w = a.anorm.bias_w; p.n_bias_b = a.anorm.bias_b;
  p.dbg = g_gemm_debug;
  p.u.hints = POL_HIDDEN << 6;  // bf16 stores of the first product's epilogue: the hidden tiles going to the scratch
  p.d.hints = 0;

  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(mlp_pair_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_pair_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(mlp_pair_kernel)");
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le = a.stats ? cudaLaunchKernelEx(&cfg, mlp_pair_kernel<true>, ta, tw1, tw2, ths, thl, tres, t32, t16, p)
                           : cudaLaunchKernelEx(&cfg, mlp_pair_kernel<false>, ta, tw1, tw2, ths, thl, tres, t32, t16, p);
  if (le != cudaSuccess) return fail_cuda(le, "mlp_pair_kernel launch");
  GECCO_CHECK_LAUNCH("mlp_pair_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco
