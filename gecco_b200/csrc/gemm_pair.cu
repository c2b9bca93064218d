// CTA-pair tcgen05 GEMM (cta_group::2) for the K <= 384 projections of the point stream (k|v|q, mlp.0, unpool
// out-proj).  Two CTAs on the SMs of one TPC work on a 256-row x 192-column tile: each CTA keeps ITS 128 rows of A
// resident in shared memory for all column blocks of the row block (6 k-blocks x 16 KB, loaded once per row block) and
// streams only HALF of every weight tile (96 rows x 64 k), because tcgen05.mma.cta_group::2 reads the B operand
// from both CTAs' shared memory.  Per 256 x 192 x 384 tile the pair pulls 144 KB of operands from L2 instead of
// 2 x 240 KB for two single-CTA tiles, which is what bounds the single-CTA kernel (L2 -> SM bandwidth).
//
//   warp 0 : TMA producer (both CTAs; byte counts complete on the leader's barriers)
//   warp 1 : MMA issuer   (leader CTA only; M=256 N=192 K=16, accumulators in both CTAs' TMEM, 2 slots)
//   warp 2 : TMEM allocator (both CTAs, collective cta_group::2 allocation)
//   warp 3 : residual loader
//   warps 4-11 : epilogue (epilogue.cuh), each CTA on its own 128 rows
//
// kANorm variant (gecco_anorm): the A operand is AdaGN(x) of the bf16 residual-stream copy, normalised on the fly.  The
// bf16 k-blocks land in the resident A tile exactly as in the plain kernel (all six in flight, each CTA on its own
// barrier); warps 2 and 3 (64 threads) then rewrite every k-block IN PLACE as  bf16(a[k] * x + s[k])  (fp32 arithmetic,
// per-cloud per-channel a = scale(t) * rstd_g, s = bias(t) - a * mean_g from the group statistics, computed one row
// block ahead) and hand it to the MMA issuer.  No normalised tensor and no per-cloud folded weights exist in HBM.
#include "common.cuh"
#include "debug_api.h"
#include "epilogue.cuh"
#include "kernels.cuh"
#include "norm.cuh"
#include "ptx.cuh"

namespace gecco {

int epi_skip_option();
long long* g_gemm_debug = nullptr;  // device buffer [grid][16] of cycle counters, set by gecco_set_debug_buffer

namespace {

constexpr int BM = 128;             // rows per CTA (256 per pair)
constexpr int BN = 192;             // columns per tile
constexpr int BNH = BN / 2;         // weight rows each CTA loads
constexpr int BK = 64;
constexpr int MAX_KB = 6;           // K <= 384
constexpr int MAX_BSTAGES = 9;      // weight ring depth is chosen per launch from the shared memory the epilogue leaves
constexpr int A_KB_BYTES = BM * BK * 2;     // 16 KiB
constexpr int B_STAGE_BYTES = BNH * BK * 2; // 12 KiB
constexpr int ACC_COLS = 256;
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 128 + EPI_GROUPS * EPI_THREADS;
constexpr int SMEM_LIMIT = 232448;
constexpr int SMEM_FIXED = MAX_KB * A_KB_BYTES + 1024 /*align*/ + 512 /*barriers*/;
constexpr int NORM_BYTES = 2 * 2 * MAX_KB * BK * 4;  // a[K], s[K], double buffered over row blocks
constexpr int ANORM_SMEM = NORM_BYTES;
constexpr int XF_THREADS = 64;              // warps 2 and 3
// L2 residency hints per launch class (bits 0-1 A loads, 2-3 residual loads, 4-5 fp32 stores, 6-7 bf16 stores; ptx.cuh
// l2_policy kinds)
constexpr int HINTS_RESIDUAL_PROJ = 160;  // residual projections (unpool out-proj): both outputs evict_last, the MLP reads them next
constexpr int HINTS_OTHER_PROJ = 0;       // normalising (k|v|q) and plain projections

struct PParams {
  EpiParams e;
  int num_kb, w_rows_per_cloud;
  int num_pair_blocks, num_n_blocks;
  int bstages;
  int kbps;  // k-blocks per weight stage: one barrier round trip of the MMA thread per kbps * 4 MMAs
  long long* dbg;  // optional [grid][16] cycle counters (gecco_set_debug_buffer), nullptr in production
  // A-operand normalisation (kANorm)
  const double* n_stats; int n_stat_gs, n_groups; float n_eps;
  const float* n_t; int n_t_stride;
  const float *n_scale_w, *n_scale_b, *n_bias_w, *n_bias_b;
  int K;
  int a_hint;  // L2 residency hint of the A-operand loads (ptx.cuh l2_policy kinds)
};

__device__ __forceinline__ int num_kb_of(const PParams& p) { return p.num_kb; }

// cycles spent in a barrier wait, accumulated into `acc` when the debug buffer is set
#define TIMED_WAIT(acc, bar, parity)        \
  do {                                      \
    if (GECCO_DBG_ON(p.dbg)) {                 \
      const long long t0__ = clock64();     \
      mbar_wait(bar, parity);               \
      acc += clock64() - t0__;              \
    } else {                                \
      mbar_wait(bar, parity);               \
    }                                       \
  } while (0)

// kEpi: 0 generic epilogue, 1 generic + AdaGN statistics, 2 fast bf16-only epilogue (epi_tile_fast), 3 fast + Gaussian activation
template <int kEpi, bool kANorm>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
gemm_pair_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w,
                 const __grid_constant__ CUtensorMap tma_res, const __grid_constant__ CUtensorMap tma_o32,
               const __grid_constant__ CUtensorMap tma_o16, const PParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                                   // [MAX_KB] resident A k-blocks
  const int BSTAGES = p.bstages;
  const int kbps = p.kbps;
  const int stage_bytes = kbps * B_STAGE_BYTES;
  const int num_st = num_kb_of(p) / kbps;
  float* sNorm = reinterpret_cast<float*>(smem + MAX_KB * A_KB_BYTES);  // kANorm: a / s vectors, group mean / rstd
  uint8_t* sB = smem + MAX_KB * A_KB_BYTES + (kANorm ? ANORM_SMEM : 0);  // [BSTAGES] weight half-tiles, kbps k-blocks each
  uint8_t* sEpi = sB + BSTAGES * stage_bytes;
  constexpr bool kStats = kEpi == 1;
  constexpr bool kFast = kEpi >= 2;
  EpiSmem es;
  uint64_t* bars;
  if constexpr (kFast) {
    es.x0 = es.x1 = es.o16 = sEpi;
    es.bias = sEpi + EPI_GROUPS * EPI_FAST_O16_BYTES;
    bars = reinterpret_cast<uint64_t*>(es.bias + EPI_BIAS_BYTES);
  } else {
    bars = reinterpret_cast<uint64_t*>(epi_smem_carve(es, sEpi, p.e.has_res, p.e.o32 != nullptr, p.e.o16 != nullptr));
  }
  uint64_t* a_full = bars;                    // [MAX_KB]   leader: both CTAs' A k-block landed
  uint64_t* a_empty = a_full + MAX_KB;        // [MAX_KB]   each CTA: last MMA reading the k-block completed
  uint64_t* b_full = a_empty + MAX_KB;        // [MAX_BSTAGES]  leader
  uint64_t* b_empty = b_full + MAX_BSTAGES;   // [MAX_BSTAGES]  each CTA
  uint64_t* acc_full = b_empty + MAX_BSTAGES; // [2]        each CTA
  uint64_t* acc_empty = acc_full + 2;         // [2]        leader: one arrival per epilogue warp of both CTAs
  es.res_full = acc_empty + 2;   // [EPI_GROUPS][2]
  es.res_empty = es.res_full + EPI_NUM_BARS / 2;
  uint64_t* a_landed = es.res_full + EPI_NUM_BARS;  // [MAX_KB] each CTA: its un-normalised k-block landed (kANorm)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(a_landed + MAX_KB);

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();  // same value, provably warp-uniform for the compiler
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader
  const uint32_t urank = uniform_u32(rank);
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int num_kb = p.num_kb;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    if (p.e.has_res) tma_prefetch_desc(&tma_res);
    if (p.e.o32 != nullptr) tma_prefetch_desc(&tma_o32);
    if (p.e.o16 != nullptr) tma_prefetch_desc(&tma_o16);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < MAX_KB; ++i) {
      // kANorm: the k-block is complete when the transform warps of BOTH CTAs have written it (2 warps each)
      mbar_init(&a_full[i], kANorm ? 2 * (XF_THREADS / 32) : 1);
      mbar_init(&a_empty[i], 1);
    }
    for (int i = 0; i < MAX_KB; ++i) mbar_init(&a_landed[i], 1);
    for (int i = 0; i < MAX_BSTAGES; ++i) {
      mbar_init(&b_full[i], 1);
      mbar_init(&b_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], 2 * EPI_GROUPS * EPI_THREADS / 32);
    }
    epi_bar_init(es);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc_pair<TMEM_COLS>(tmem_slot);
  tc_fence_before_sync();
  cluster_sync_all();  // barriers of both CTAs are initialised before any remote arrive / TMA completion
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch_dependents();

  // warps 0-3 (TMA / MMA / allocator / residual loader: a handful of registers) hand their registers to the epilogue
  if (warp < 4) {
  setmaxnreg_dec<kANorm ? 104 : 40>();
  if (warp == 0 && lane == 0) {
    // ------------------------------------------------------------ TMA producer (both CTAs)
    int stage = 0;
    uint32_t bphase = 0;
    uint32_t it = 0;
    long long w_aempty = 0, w_bempty = 0;
    const long long t_start = clock64();
    const uint64_t a_pol = l2_policy(p.a_hint);
    for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
      const int m0 = pb * 2 * BM + (int)rank * BM;
      const int cloud_w = p.w_rows_per_cloud ? (m0 / p.e.rows_per_cloud) * p.w_rows_per_cloud : 0;
      for (int nb = 0; nb < p.num_n_blocks; ++nb) {
        const int wrow = cloud_w + nb * BN + (int)rank * BNH;
        for (int st = 0; st < num_st; ++st) {
          TIMED_WAIT(w_bempty, &b_empty[stage], bphase ^ 1u);
          if (rank == 0) mbar_arrive_expect_tx(&b_full[stage], 2 * stage_bytes);
          for (int kk = 0; kk < kbps; ++kk) {
            const int kb = st * kbps + kk;
            if (nb == 0) {
              if constexpr (kANorm) {
                // the un-normalised k-block lands on this CTA's own barrier; the transform warps rewrite it in place and
                // then complete the leader's a_full[kb]
                TIMED_WAIT(w_aempty, &a_empty[kb], (it & 1u) ^ 1u);
                mbar_arrive_expect_tx(&a_landed[kb], A_KB_BYTES);
                tma_load_2d_h(sA + kb * A_KB_BYTES, &tma_a, &a_landed[kb], kb * BK, m0, a_pol);
              } else {
                // this CTA's 128 rows of A, k-block kb: resident for all column blocks of the row block
                TIMED_WAIT(w_aempty, &a_empty[kb], (it & 1u) ^ 1u);
                if (rank == 0) mbar_arrive_expect_tx(&a_full[kb], 2 * A_KB_BYTES);
                tma_load_2d_pair_h(sA + kb * A_KB_BYTES, &tma_a, &a_full[kb], kb * BK, m0, a_pol);
              }
            }
            tma_load_2d_pair(sB + stage * stage_bytes + kk * B_STAGE_BYTES, &tma_w, &b_full[stage], kb * BK, wrow);
          }
          if (++stage == BSTAGES) { stage = 0; bphase ^= 1u; }
        }
      }
    }
    if (GECCO_DBG_ON(p.dbg)) {
      long long* d = p.dbg + (long long)blockIdx.x * 32;
      d[0] = clock64() - t_start; d[1] = w_aempty; d[2] = w_bempty;
    }
  } else if (uwarp == 1) {
    // ------------------------------------------------------------ MMA issuer (leader CTA): the whole warp runs the loop
    // (uniform control flow keeps the descriptors in uniform registers), one elected lane issues
    if (urank == 0) {
      constexpr uint32_t idesc = umma_idesc_bf16(2 * BM, BN);
      const uint32_t sA_u = uniform_u32(smem_u32(sA)), sB_u = uniform_u32(smem_u32(sB));
      const uint32_t tmem_u = uniform_u32(tmem_base);
      int stage = 0;
      uint32_t bphase = 0;
      uint32_t it = 0, tile = 0;
      long long w_acc = 0, w_afull = 0, w_bfull = 0, w_issue = 0;
      const long long t_start = clock64();
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
        for (int nb = 0; nb < p.num_n_blocks; ++nb, ++tile) {
          const uint32_t slot = tile & 1u;
          TIMED_WAIT(w_acc, &acc_empty[slot], ((tile >> 1) & 1u) ^ 1u);
          tc_fence_after_sync();
          const uint32_t tmem_d = tmem_u + slot * ACC_COLS;
          const bool last_nb = nb == p.num_n_blocks - 1;
          for (int st = 0; st < num_st; ++st) {
            TIMED_WAIT(w_bfull, &b_full[stage], bphase);
            for (int kk = 0; kk < kbps; ++kk) {
              const int kb = st * kbps + kk;
              if (nb == 0) TIMED_WAIT(w_afull, &a_full[kb], it & 1u);
              tc_fence_after_sync();
              const uint64_t da = umma_desc_k_sw128(sA_u + kb * A_KB_BYTES);
              const uint64_t db = umma_desc_k_sw128(sB_u + stage * stage_bytes + kk * B_STAGE_BYTES);
              long long ti0 = 0;
              if (GECCO_DBG_ON(p.dbg)) ti0 = clock64();
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_bf16_ss_pair(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
                if (last_nb) umma_commit_pair(&a_empty[kb]);  // the k-block may be reloaded for the next row block
              }
              __syncwarp();
              if (GECCO_DBG_ON(p.dbg)) w_issue += clock64() - ti0;
            }
            if (elect_one()) umma_commit_pair(&b_empty[stage]);
            __syncwarp();
            if (++stage == BSTAGES) { stage = 0; bphase ^= 1u; }
          }
          if (elect_one()) umma_commit_pair(&acc_full[slot]);
          __syncwarp();
        }
      }
      if (GECCO_DBG_ON(p.dbg) && lane == 0) {
        long long* d = p.dbg + (long long)blockIdx.x * 32;
        d[3] = clock64() - t_start; d[4] = w_acc; d[5] = w_afull; d[6] = w_bfull; d[7] = tile; d[12] = w_issue;
      }
    }
  } else if (kANorm && (uwarp == 2 || uwarp == 3)) {
    // ------------------------------------------------------------ A-operand transform: AdaGN in place on the resident k-blocks
    // A quarter warp owns one 128-byte row per access (eight 16-byte chunks: conflict free under any swizzle); a thread
    // keeps physical chunk j = tt & 7 of rows  (tt >> 3) + 8 i,  whose low three bits never change, so the LOGICAL chunk
    // j ^ (row & 7) -- the eight channels it normalises -- is fixed and their a / s stay in 16 registers per k-block.
    const int tt = threadIdx.x - 64;             // 0..63
    const uint32_t pj = (uint32_t)tt & 7u, rl = (uint32_t)tt >> 3;
    const uint32_t lj = pj ^ rl;                 // logical chunk: channels 8 lj .. 8 lj + 7 of the k-block
    const int K = p.K, gs = K / p.n_groups;
    const double count = (double)p.e.valid_rows * gs;
    // a / s of a row block from the group statistics, computed one row block ahead.  FP64 division and square root cost
    // thousands of cycles per warp on this part, so the double-precision work is two multiplies and one FMA per channel
    // (mean = s1 / n and E[x^2] - mean^2 need the precision, rstd does not) and the statistics loads are issued first.
    const double inv_count = 1.0 / count;
    auto make_norm = [&](int pb, uint32_t buf) {
      const int m0 = pb * 2 * BM + (int)rank * BM;
      const int cloud = m0 / p.e.rows_per_cloud;
      const double* cst = p.n_stats + (long long)cloud * (K / p.n_stat_gs) * 2;
      float* na = sNorm + buf * 2 * MAX_KB * BK;
      float* ns = na + MAX_KB * BK;
      const float tc = __ldg(p.n_t + (long long)cloud * p.n_t_stride);
      const int per = gs / p.n_stat_gs;
      // all global loads of this thread's channels first (MAX_KB * BK / XF_THREADS = 6), then the arithmetic: one L2
      // round trip instead of six
      constexpr int NCH = MAX_KB * BK / XF_THREADS;
      double s1[NCH], s2[NCH];
      float sw[NCH], sb[NCH], bw[NCH], bb[NCH];
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = tt + i * XF_THREADS;
        s1[i] = s2[i] = 0.0;
        sw[i] = sb[i] = bw[i] = bb[i] = 0.f;
        if (c < K) {
          const int g = c / gs;
          for (int j = 0; j < per; ++j) {
            s1[i] += cst[(g * per + j) * 2];
            s2[i] += cst[(g * per + j) * 2 + 1];
          }
          sw[i] = __ldg(p.n_scale_w + c); sb[i] = __ldg(p.n_scale_b + c);
          bw[i] = __ldg(p.n_bias_w + c); bb[i] = __ldg(p.n_bias_b + c);
        }
      }
#pragma unroll
      for (int i = 0; i < NCH; ++i) {
        const int c = tt + i * XF_THREADS;
        if (c < K) {
          const double m = s1[i] * inv_count;
          double var = fma(-m, m, s2[i] * inv_count);
          if (var < 0.0) var = 0.0;
          const float rstd = rsqrtf(static_cast<float>(var) + p.n_eps);
          const float a = (tc * sw[i] + sb[i]) * rstd;
          na[c] = a;
          ns[c] = (tc * bw[i] + bb[i]) - a * static_cast<float>(m);
        }
      }
      named_bar_sync(2, XF_THREADS);  // a / s visible to both warps
    };
    uint32_t it = 0;
    const uint32_t row0 = smem_u32(sA) + rl * 128u + (pj << 4);  // this thread's chunk of row rl of k-block 0
    long long x_aempty = 0, x_stg = 0, x_norm = 0;
    const long long x_start = clock64();
    if (pair < p.num_pair_blocks) make_norm(pair, 0);
    for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
      const uint32_t na_u = smem_u32(sNorm + (it & 1u) * 2 * MAX_KB * BK), ns_u = na_u + MAX_KB * BK * 4;
      for (int kb = 0; kb < num_kb; ++kb) {
        const uint32_t ko = (uint32_t)(kb * BK) * 4u + lj * 32u;
        const float4 a0 = lds128(na_u + ko), a1 = lds128(na_u + ko + 16u);
        const float4 s0 = lds128(ns_u + ko), s1 = lds128(ns_u + ko + 16u);
        TIMED_WAIT(x_stg, &a_landed[kb], it & 1u);
        const uint32_t base = row0 + kb * A_KB_BYTES;
#pragma unroll
        for (int b = 0; b < 2; ++b) {  // eight rows (eight LDS.128) in flight
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
        fence_proxy_async_smem();  // generic-proxy writes of the k-block -> visible to the tensor core's reads
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(&a_full[kb]);
      }
      // a / s of the next row block, off the critical path (the tile is resident for several column blocks now)
      long long xn0 = 0;
      if (GECCO_DBG_ON(p.dbg)) xn0 = clock64();
      if (pb + num_pairs < p.num_pair_blocks) make_norm(pb + num_pairs, (it & 1u) ^ 1u);
      if (GECCO_DBG_ON(p.dbg)) x_norm += clock64() - xn0;
    }
    if (GECCO_DBG_ON(p.dbg) && tt == 0) {
      long long* d = p.dbg + (long long)blockIdx.x * 32;
      d[22] = clock64() - x_start; d[23] = x_aempty; d[24] = x_stg; d[25] = x_norm;
    }
  } else if (warp == 3 && lane == 0) {
    // ------------------------------------------------------------ residual loader
    if (p.e.has_res && !(p.e.skip & 2)) {
      uint32_t cnt[EPI_GROUPS] = {0, 0};
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs) {
        const int m0 = pb * 2 * BM + (int)rank * BM;
        for (int nb = 0; nb < p.num_n_blocks; ++nb) epi_load_residual_panel(p.e, es, &tma_res, m0, nb * BN, cnt);
      }
    }
  }
  } else {
    setmaxnreg_inc<kANorm ? 200 : 232>();
    // ------------------------------------------------------------ epilogue (each CTA: its own 128 rows)
    const EpiThread et = epi_thread_init(es, (warp - 4) >> 2, threadIdx.x & (EPI_THREADS - 1));
    const int q = warp & 3;
    uint32_t tile = 0, cnt = 0;
    long long w_accfull = 0, w_pref = 0;
    const long long t_start = clock64();
    EpiBias bias_r;
    if (pair < p.num_pair_blocks) epi_bias_load(p.e, et, pair * 2 * BM + (int)rank * BM, 0, bias_r);
    for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs) {
      const int m0 = pb * 2 * BM + (int)rank * BM;
      for (int nb = 0; nb < p.num_n_blocks; ++nb, ++tile) {
        const uint32_t slot = tile & 1u;
        long long tp0 = 0;
        if (GECCO_DBG_ON(p.dbg)) tp0 = clock64();
        epi_bias_stage(p.e, et, bias_r);
        // the next panel's bias is loaded under this panel
        if (nb + 1 < p.num_n_blocks) epi_bias_load(p.e, et, m0, (nb + 1) * BN, bias_r);
        else if (pb + num_pairs < p.num_pair_blocks) epi_bias_load(p.e, et, (pb + num_pairs) * 2 * BM + (int)rank * BM, 0, bias_r);
        if (GECCO_DBG_ON(p.dbg)) w_pref += clock64() - tp0;
        TIMED_WAIT(w_accfull, &acc_full[slot], (tile >> 1) & 1u);
        tc_fence_after_sync();
        const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot * ACC_COLS;
        if constexpr (kFast) {
          // a 128-row tile lies inside one cloud (rows_per_cloud % 256 == 0)
          const bool row_valid = (m0 % p.e.rows_per_cloud) + q * 32 + (int)et.lane < p.e.valid_rows;
          epi_tile_fast<kEpi == 3>(p.e, et, &tma_o16, taddr, m0, nb * BN, smem_u32(es.o16), row_valid, [&] {
            tc_fence_before_sync();
            __syncwarp();
            if (et.lane == 0) mbar_arrive_leader(&acc_empty[slot]);  // one (remote) arrival per warp
          });
        } else {
          epi_panel<kStats>(p.e, es, et, &tma_o32, &tma_o16, taddr, m0, nb * BN, cnt);
          tc_fence_before_sync();
          __syncwarp();
          if (et.lane == 0) mbar_arrive_leader(&acc_empty[slot]);  // one (remote) arrival per warp
        }
      }
    }
    if (et.lane == 0) tma_store_wait_read<0>();
    if (GECCO_DBG_ON(p.dbg) && et.lane == 0 && et.q == 0) {
      long long* d = p.dbg + (long long)blockIdx.x * 32 + 8 + 2 * et.grp;
      d[0] = clock64() - t_start; d[1] = w_accfull;
      if (et.grp == 0) p.dbg[(long long)blockIdx.x * 32 + 15] = w_pref;
    }
  }

  // the peer's shared memory and barriers must stay valid until the leader's last MMA / commit has completed
  tc_fence_before_sync();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc_pair<TMEM_COLS>(tmem_base);
  }
}

}  // namespace

// gecco_set_option("fast_epilogue", 0): the generic epilogue everywhere (A/B measurements, tests)
static bool g_fast_epilogue = true;
void set_fast_epilogue_option(int value) { g_fast_epilogue = value != 0; }

bool gemm_pair_shape_ok(int m, int rows_per_cloud, int n_out, int k) {
  if (k > MAX_KB * BK || k % 8 != 0 || m % (2 * BM) != 0 || m < 2 * BM * 8 || sm_count() < 2) return false;
  if (rows_per_cloud % (2 * BM) != 0) return false;
  return n_out % BNH == 0;  // every CTA of the pair owns a full half tile of weight rows
}

bool gemm_anorm_supported(int m, int rows_per_cloud, int n_out, int k) {
  return g_use_pairs_ref() && gemm_pair_shape_ok(m, rows_per_cloud, n_out, k) && k % BK == 0;
}

int launch_gemm_pair(const gecco_gemm_args& a, cudaStream_t stream, int* handled) {
  *handled = 0;
  const int sms = sm_count();
  if (!gemm_pair_shape_ok(a.m, a.rows_per_cloud, a.n_out, a.k)) return GECCO_OK;
  const bool anorm = a.anorm.stats != nullptr;
  if (anorm) {
    GECCO_REQUIRE(a.k % BK == 0, "gemm: A-operand normalisation needs k %% 64 == 0 (got %d)", a.k);
    GECCO_REQUIRE(a.res == nullptr, "gemm: A-operand normalisation cannot be combined with a residual");
    GECCO_REQUIRE(a.anorm.t && a.anorm.scale_w && a.anorm.scale_b && a.anorm.bias_w && a.anorm.bias_b,
                  "gemm: incomplete A-operand normalisation (t / scale / bias)");
    GECCO_REQUIRE(a.anorm.groups <= 128, "gemm: A-operand normalisation supports at most 128 groups");
    GECCO_REQUIRE(a.anorm.groups > 0 && a.k % a.anorm.groups == 0 && a.anorm.stat_gs > 0 &&
                      (a.k / a.anorm.groups) % a.anorm.stat_gs == 0,
                  "gemm: A-operand normalisation groups (%d) / statistics granularity (%d) do not fit k = %d", a.anorm.groups,
                  a.anorm.stat_gs, a.k);
  }

  const int clouds = ceil_div(a.m, a.rows_per_cloud);
  const uint64_t w_rows = a.w_rows_per_cloud ? (uint64_t)a.w_rows_per_cloud * (clouds - 1) + a.n_out : (uint64_t)a.n_out;
  CUtensorMap ta, tw, tres, t32, t16;
  if (int rc = make_tmap_bf16(&ta, a.a, a.k, a.m, a.lda, BM)) return rc;
  if (int rc = make_tmap_bf16(&tw, a.w, a.k, w_rows, a.ldw, BNH)) return rc;
  if (int rc = make_residual_tmap(a.res, a.ldr, a.m, a.n_out, ta, &tres)) return rc;
  if (int rc = make_output_tmaps(a.out_f32, a.ldo32, a.out_bf16, a.ldo16, a.m, a.n_out, ta, &t32, &t16)) return rc;

  PParams p;
  p.e.M = a.m; p.e.n_out = a.n_out;
  p.e.rows_per_cloud = a.rows_per_cloud; p.e.valid_rows = a.valid_rows;
  p.e.bias = a.bias; p.e.bias_stride = a.bias_stride;
  p.e.act = a.act;
  p.e.act_k = a.act ? static_cast<float>(-1.4426950408889634 / (2.0 * (double)a.act_alpha * (double)a.act_alpha)) : 0.f;
  p.e.has_res = a.res != nullptr;
  p.e.o32 = a.out_f32;
  p.e.o16 = static_cast<__nv_bfloat16*>(a.out_bf16);
  p.e.stats = a.stats;
  p.e.geom = a.geom; p.e.sigma = a.sigma; p.e.sigma_stride = a.sigma_stride; p.e.sigma_data = a.sigma_data; p.e.wx = a.wx;
  p.num_kb = ceil_div(a.k, BK);
  p.w_rows_per_cloud = a.w_rows_per_cloud;
  p.num_pair_blocks = a.m / (2 * BM);
  p.num_n_blocks = ceil_div(a.n_out, BN);
  p.dbg = g_gemm_debug;
  p.e.dbg = g_gemm_debug;
  p.e.skip = epi_skip_option();
  p.e.hints = a.res != nullptr ? HINTS_RESIDUAL_PROJ : HINTS_OTHER_PROJ;
  p.a_hint = p.e.hints & 3;
  p.n_stats = a.anorm.stats; p.n_stat_gs = a.anorm.stat_gs; p.n_groups = a.anorm.groups; p.n_eps = a.anorm.eps;
  p.n_t = a.anorm.t; p.n_t_stride = a.anorm.t_stride;
  p.n_scale_w = a.anorm.scale_w; p.n_scale_b = a.anorm.scale_b; p.n_bias_w = a.anorm.bias_w; p.n_bias_b = a.anorm.bias_b;
  p.K = a.k;
  // bf16-only whole-tile projections take the fast epilogue
  const bool fast = g_fast_epilogue && a.res == nullptr && a.stats == nullptr && a.out_f32 == nullptr && a.geom == nullptr &&
                    a.bias != nullptr && a.out_bf16 != nullptr && a.n_out % BN == 0 &&
                    p.e.skip == 0;
  const int epi_bytes = (fast ? epi_fast_smem_bytes() : epi_smem_bytes(p.e.has_res, a.out_f32 != nullptr, a.out_bf16 != nullptr)) +
                        (anorm ? ANORM_SMEM : 0);
  const int avail = SMEM_LIMIT - SMEM_FIXED - epi_bytes;
  p.kbps = 1;
  for (int cand = p.num_kb; cand > 1; --cand)  // deepest weight stage that still leaves a 3-deep ring
    if (p.num_kb % cand == 0 && avail / (cand * B_STAGE_BYTES) >= 3) { p.kbps = cand; break; }
  p.bstages = avail / (p.kbps * B_STAGE_BYTES);
  if (p.bstages > MAX_BSTAGES) p.bstages = MAX_BSTAGES;
  GECCO_REQUIRE(p.bstages >= 2, "gemm_pair: shared memory budget");
  const int smem_bytes = SMEM_FIXED + epi_bytes + p.bstages * p.kbps * B_STAGE_BYTES;

  using KernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, PParams);
  static const KernelFn kernels[4][2] = {{gemm_pair_kernel<0, false>, gemm_pair_kernel<0, true>},
                                         {gemm_pair_kernel<1, false>, gemm_pair_kernel<1, true>},
                                         {gemm_pair_kernel<2, false>, gemm_pair_kernel<2, true>},
                                         {gemm_pair_kernel<3, false>, gemm_pair_kernel<3, true>}};
  static bool attr_set = false;
  if (!attr_set) {
    for (int i = 0; i < 4; ++i)
      for (int j = 0; j < 2; ++j) {
        cudaError_t e = cudaFuncSetAttribute(kernels[i][j], cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
        if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(gemm_pair_kernel)");
      }
    attr_set = true;
  }
  const int epi_kind = fast ? (a.act ? 3 : 2) : (a.stats ? 1 : 0);
  int pairs = sms / 2;
  if (pairs > p.num_pair_blocks) pairs = p.num_pair_blocks;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le = cudaLaunchKernelEx(&cfg, kernels[epi_kind][anorm ? 1 : 0], ta, tw, tres, t32, t16, p);
  if (le != cudaSuccess) return fail_cuda(le, "gemm_pair_kernel launch");
  GECCO_CHECK_LAUNCH("gemm_pair_kernel launch");
  *handled = 1;
  return GECCO_OK;
}

}  // namespace gecco

/* Development aid: a device buffer of at least 148 * 16 int64 receiving per-CTA cycle counters of the pair GEMM
 * ([0] producer total, [1] wait A free, [2] wait W stage free, [3] MMA total, [4] wait accumulator free, [5] wait A landed,
 * [6] wait W landed, [7] tiles, [8],[10] epilogue group total, [9],[11] epilogue wait accumulator).  NULL disables it. */
extern "C" int gecco_set_debug_buffer(void* buf) {
  gecco::g_gemm_debug = static_cast<long long*>(buf);
  return GECCO_OK;
}
