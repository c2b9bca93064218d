// Fused point-side MLP of a BroadcastingLayer (models/set_transformer.py:165-166, models/mlp.py:5-39,
// models/activation.py:17-24):
//     x <- x + W2 . g(W1_b . xb + b1_b) + b2          (W1_b, b1_b: mlp.0 with AdaGN_mlp folded in per cloud)
// as ONE tcgen05 kernel.  The 768-wide hidden activation never leaves the SM: it is produced in 128-column chunks in
// TMEM, pulled into registers by the epilogue warps (which frees the TMEM buffer for the next chunk at once), passed
// through the Gaussian activation, written as bf16 into shared memory in the UMMA K-major 128B-swizzled layout and
// consumed as the A operand of the second GEMM, whose 128 x 384 fp32 accumulator stays in TMEM for the whole row
// block.  Compared with the two-GEMM path this removes one write and one read of the [rows, 768] bf16 hidden tensor
// per layer (402 MB at 64 clouds x 2048 points).
//
// CTA pair (cta_group::2), 256 rows per pair, 128 per CTA.  TMEM (512 columns per CTA):
//     [0, 384)   Y   accumulator of the second GEMM (two N=192 halves)
//     [384, 512) H   accumulator of the first GEMM for one 128-column hidden chunk
// Shared memory per CTA: A row block resident (6 x 16 KB), one bf16 hidden chunk (2 k-blocks x 16 KB, reused as the
// fp32 output staging of the final epilogue), W1 ring (4 x 8 KB: 64 weight rows x 64 k per CTA), W2 ring (2 x 12 KB:
// 96 weight rows x 64 k per CTA, reused as the bf16 output staging), residual chunks (2 x 16 KB).
//
//   warp 0 : TMA producer for A and W1          warp 2 : TMEM allocator, then TMA producer for W2
//   warp 1 : MMA issuer (leader CTA)            warp 3 : residual loader
//   warps 4-11 : activation of the hidden chunks, then the final epilogue (epilogue.cuh) of the row block
//
// MMA issue order over the chunks g = 0, 1, ... of all row blocks of the pair: G1(0), then per chunk
// { G1(g+1) once the activation warps hold H(g) in registers;  G2(g) once the bf16 chunk is in shared memory },
// so the first GEMM of the next chunk (or of the next row block) runs under the activation of the current one and
// under the final epilogue.
#include "common.cuh"
#include "epilogue.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace gecco {
int epi_skip_option();
extern long long* g_gemm_debug;  // gemm_pair.cu: optional [grid][32] cycle counters (gecco_set_debug_buffer)
namespace {

// cycles spent in `stmt`, accumulated into `acc` when the debug buffer is set
#define TIMED(acc, stmt)                    \
  do {                                      \
    if (GECCO_DBG_ON(p.dbg)) {                 \
      const long long t0__ = clock64();     \
      stmt;                                 \
      acc += clock64() - t0__;              \
    } else {                                \
      stmt;                                 \
    }                                       \
  } while (0)

constexpr int BM = 128;              // rows per CTA (256 per pair)
constexpr int C = 384;               // feature width (= K of GEMM 1 = N of GEMM 2)
constexpr int BK = 64;
constexpr int NKB = C / BK;          // 6 k-blocks of A
constexpr int HC = 128;              // hidden columns per chunk
constexpr int HKB = HC / BK;         // k-blocks of the second GEMM per chunk
constexpr int A_KB_BYTES = BM * BK * 2;        // 16 KiB
constexpr int H_KB_BYTES = BM * BK * 2;        // 16 KiB: 128 rows x 64 hidden columns
constexpr int W1_SLOT = (HC / 2) * BK * 2;     // 8 KiB: 64 rows of W1 x 64 k
constexpr int W2_ROWS = 96;                    // rows of W2 per CTA per N=192 half
constexpr int W2_SLOT = W2_ROWS * BK * 2;      // 12 KiB
constexpr int W1_SLOTS = 4;
constexpr int W2_SLOTS = 2;
constexpr int Y_COLS = C;
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 128 + EPI_GROUPS * EPI_THREADS;
constexpr int EPI_WARPS = EPI_GROUPS * EPI_THREADS / 32;  // 8
constexpr int SMEM_BYTES = 1024 /*align*/ + NKB * A_KB_BYTES + HKB * H_KB_BYTES + W1_SLOTS * W1_SLOT + W2_SLOTS * W2_SLOT +
                           EPI_GROUPS * EPI_RES_BYTES + EPI_BIAS_BYTES + 512 /*barriers*/;
static_assert(HKB * H_KB_BYTES == EPI_GROUPS * EPI_RES_BYTES, "the second residual / output buffers alias the hidden chunk buffer");
static_assert((C / EPI_CHUNK / EPI_GROUPS) % 2 == 0, "every group must start a row block on its first buffer");
static_assert(W2_SLOTS * W2_SLOT >= EPI_GROUPS * EPI_O16_BYTES, "the bf16 output staging aliases the W2 ring");
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct MParams {
  EpiParams e;                 // final epilogue: + b2, + residual, statistics, fp32 / bf16 stores
  const float* b1;             // [clouds][b1_stride] (folded) or [hidden]
  int b1_stride;
  float act_k;                 // -log2(e) / (2 alpha^2)
  int w1_rows_per_cloud;
  int num_chunks;              // hidden / 128
  int num_pair_blocks;
  long long* dbg;              // development aid, nullptr in production
};

__device__ __forceinline__ float gauss_act(float v, float k) {
  return fmaf(ex2_approx(v * v * k), 1.0f / 0.28f, -0.7f / 0.28f);
}

template <bool kStats>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
mlp_fused_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w1,
                 const __grid_constant__ CUtensorMap tma_w2, const __grid_constant__ CUtensorMap tma_res,
                 const __grid_constant__ CUtensorMap tma_o32, const __grid_constant__ CUtensorMap tma_o16, const MParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sA = smem;                               // [NKB] resident A k-blocks
  uint8_t* sH = sA + NKB * A_KB_BYTES;              // [HKB] bf16 hidden chunk | fp32 output staging of the epilogue
  uint8_t* sW1 = sH + HKB * H_KB_BYTES;             // [W1_SLOTS]
  uint8_t* sW2 = sW1 + W1_SLOTS * W1_SLOT;          // [W2_SLOTS] | bf16 output staging of the epilogue
  uint8_t* sE = sW2 + W2_SLOTS * W2_SLOT;
  EpiSmem es;
  es.x0 = sE;    // residual / fp32 output staging, first buffer of each group: dedicated, so the loader can run ahead
  es.x1 = sH;    // second buffer of each group: the hidden chunk buffer, free once Y is complete
  es.o16 = sW2;
  es.bias = sE + EPI_GROUPS * EPI_RES_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(es.bias + EPI_BIAS_BYTES);
  uint64_t* a_full = bars;                       // [NKB]       leader
  uint64_t* a_empty = a_full + NKB;              // [1]         each CTA: the last first-GEMM of the row block is complete
  uint64_t* w1_full = a_empty + 1;               // [W1_SLOTS]  leader
  uint64_t* w1_empty = w1_full + W1_SLOTS;       // [W1_SLOTS]  each CTA
  uint64_t* w2_full = w1_empty + W1_SLOTS;       // [W2_SLOTS]  leader
  uint64_t* w2_empty = w2_full + W2_SLOTS;       // [W2_SLOTS]  each CTA
  uint64_t* h_full = w2_empty + W2_SLOTS;        // [1] each CTA: first GEMM of the chunk complete (TMEM H)
  uint64_t* h_free = h_full + 1;                 // [1] leader: TMEM H is in registers in both CTAs (one arrival per warp)
  uint64_t* h_ready = h_free + 1;                // [1] leader: bf16 chunk in both CTAs' smem (one arrival per warp)
  uint64_t* hc_empty = h_ready + 1;              // [1] each CTA: second GEMM finished reading the smem chunk
  uint64_t* y_full = hc_empty + 1;               // [1] each CTA
  uint64_t* y_empty = y_full + 1;                // [1] leader: one arrival per epilogue warp of both CTAs
  uint64_t* epi_done = y_empty + 1;              // [1] each CTA: output staging (hidden chunk buffer, W2 ring) is free again
  es.res_full = epi_done + 1;                    // [EPI_GROUPS][2]
  es.res_empty = es.res_full + EPI_NUM_BARS / 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(es.res_full + EPI_NUM_BARS);

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();  // same value, provably warp-uniform (all threads converged here)
  const int lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();  // 0 = leader
  const uint32_t urank = uniform_u32(rank);
  const int pair = blockIdx.x >> 1;
  const int num_pairs = gridDim.x >> 1;
  const int nch = p.num_chunks;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w1);
    tma_prefetch_desc(&tma_w2);
    tma_prefetch_desc(&tma_res);
    tma_prefetch_desc(&tma_o32);
    tma_prefetch_desc(&tma_o16);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < NKB; ++i) mbar_init(&a_full[i], 1);
    mbar_init(a_empty, 1);
    for (int i = 0; i < W1_SLOTS; ++i) { mbar_init(&w1_full[i], 1); mbar_init(&w1_empty[i], 1); }
    for (int i = 0; i < W2_SLOTS; ++i) { mbar_init(&w2_full[i], 1); mbar_init(&w2_empty[i], 1); }
    mbar_init(h_full, 1);
    mbar_init(h_free, 2 * EPI_WARPS);
    mbar_init(h_ready, 2 * EPI_WARPS);
    mbar_init(hc_empty, 1);
    mbar_init(y_full, 1);
    mbar_init(y_empty, 2 * EPI_WARPS);
    mbar_init(epi_done, EPI_WARPS);
    epi_bar_init(es);
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
    setmaxnreg_dec<40>();
    if (warp == 0 && lane == 0) {
      // ------------------------------------------------------------ TMA producer: A row block + W1 (both CTAs)
      int slot = 0;
      uint32_t phase = 0, it = 0;
      long long c_a = 0, c_w1 = 0;
      const long long t_start = clock64();
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
        const int m0 = pb * 2 * BM + (int)rank * BM;
        const int w1_row0 = (p.w1_rows_per_cloud ? (m0 / p.e.rows_per_cloud) * p.w1_rows_per_cloud : 0) + (int)rank * (HC / 2);
        TIMED(c_a, mbar_wait(a_empty, (it & 1u) ^ 1u));
        for (int j = 0; j < nch; ++j) {
          for (int kb = 0; kb < NKB; ++kb) {
            if (j == 0) {
              if (rank == 0) mbar_arrive_expect_tx(&a_full[kb], 2 * A_KB_BYTES);
              tma_load_2d_pair(sA + kb * A_KB_BYTES, &tma_a, &a_full[kb], kb * BK, m0);
            }
            TIMED(c_w1, mbar_wait(&w1_empty[slot], phase ^ 1u));
            if (rank == 0) mbar_arrive_expect_tx(&w1_full[slot], 2 * W1_SLOT);
            tma_load_2d_pair(sW1 + slot * W1_SLOT, &tma_w1, &w1_full[slot], kb * BK, w1_row0 + j * HC);
            if (++slot == W1_SLOTS) { slot = 0; phase ^= 1u; }
          }
        }
      }
      if (GECCO_DBG_ON(p.dbg)) {
        long long* d = p.dbg + (long long)blockIdx.x * 32;
        d[0] = clock64() - t_start; d[1] = c_a; d[2] = c_w1;
      }
    } else if (warp == 2 && lane == 0) {
      // ------------------------------------------------------------ TMA producer: W2 (both CTAs)
      int slot = 0;
      uint32_t phase = 0, it = 0;
      long long c_w2 = 0;
      for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
        // the W2 ring doubles as the bf16 output staging of the previous row block's epilogue
        TIMED(c_w2, mbar_wait(epi_done, (it & 1u) ^ 1u));
        for (int c = 0; c < nch * HKB; ++c) {
          for (int h = 0; h < 2; ++h) {
            TIMED(c_w2, mbar_wait(&w2_empty[slot], phase ^ 1u));
            if (rank == 0) mbar_arrive_expect_tx(&w2_full[slot], 2 * W2_SLOT);
            tma_load_2d_pair(sW2 + slot * W2_SLOT, &tma_w2, &w2_full[slot], c * BK, h * (2 * W2_ROWS) + (int)rank * W2_ROWS);
            if (++slot == W2_SLOTS) { slot = 0; phase ^= 1u; }
          }
        }
      }
      if (GECCO_DBG_ON(p.dbg)) p.dbg[(long long)blockIdx.x * 32 + 3] = c_w2;
    } else if (uwarp == 1) {
      // ------------------------------------------------------------ MMA issuer (leader CTA): the whole warp runs the
      // loops (uniform control flow keeps the descriptors in uniform registers, see ptx.cuh), one elected lane issues
      if (urank == 0) {
        const uint32_t sA_u = uniform_u32(smem_u32(sA)), sH_u = uniform_u32(smem_u32(sH));
        const uint32_t sW1_u = uniform_u32(smem_u32(sW1)), sW2_u = uniform_u32(smem_u32(sW2));
        const uint32_t tmem_u = uniform_u32(tmem_base);
        constexpr uint32_t idesc1 = umma_idesc_bf16(2 * BM, HC);
        constexpr uint32_t idesc2 = umma_idesc_bf16(2 * BM, 2 * W2_ROWS);
        const uint32_t tmem_h = tmem_u + Y_COLS;
        int my_blocks = 0;
        for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs) ++my_blocks;
        const uint32_t total = (uint32_t)my_blocks * (uint32_t)nch;
        int s1 = 0, s2 = 0;
        uint32_t ph1 = 0, ph2 = 0;
        long long c_w1f = 0, c_af = 0, c_hf = 0, c_hr = 0, c_ye = 0, c_w2f = 0;
        const long long t_start = clock64();
        // first GEMM of global chunk g (chunk j = g % nch of the pair's row block g / nch): H = A . W1[chunk j]^T
        auto first_gemm = [&](uint32_t g) {
          const uint32_t blk = g / (uint32_t)nch, j = g % (uint32_t)nch;
          for (int kb = 0; kb < NKB; ++kb) {
            TIMED(c_w1f, mbar_wait(&w1_full[s1], ph1));
            if (j == 0) TIMED(c_af, mbar_wait(&a_full[kb], blk & 1u));
            tc_fence_after_sync();
            const uint64_t da = umma_desc_k_sw128(sA_u + kb * A_KB_BYTES);
            const uint64_t db = umma_desc_k_sw128(sW1_u + s1 * W1_SLOT);
            if (elect_one()) {
#pragma unroll
              for (int k = 0; k < BK / 16; ++k) umma_bf16_ss_pair(tmem_h, da + 2 * k, db + 2 * k, idesc1, (kb | k) ? 1u : 0u);
              umma_commit_pair(&w1_empty[s1]);
            }
            __syncwarp();
            if (++s1 == W1_SLOTS) { s1 = 0; ph1 ^= 1u; }
          }
          if (elect_one()) {
            if (j == (uint32_t)nch - 1) umma_commit_pair(a_empty);  // the A row block may be replaced
            umma_commit_pair(h_full);
          }
          __syncwarp();
        };
        first_gemm(0);
        for (uint32_t g = 0; g < total; ++g) {
          const uint32_t blk = g / (uint32_t)nch, j = g % (uint32_t)nch;
          if (g + 1 < total) {
            TIMED(c_hf, mbar_wait(h_free, g & 1u));  // H(g) is in registers: its TMEM buffer may be overwritten
            tc_fence_after_sync();
            first_gemm(g + 1);
          }
          // second GEMM of chunk g: Y (+)= Hbf16[chunk j] . W2[:, chunk j]^T
          TIMED(c_hr, mbar_wait(h_ready, g & 1u));
          if (j == 0) TIMED(c_ye, mbar_wait(y_empty, (blk & 1u) ^ 1u));
          tc_fence_after_sync();
          for (int kb = 0; kb < HKB; ++kb) {
            const uint64_t da = umma_desc_k_sw128(sH_u + kb * H_KB_BYTES);
            for (int h = 0; h < 2; ++h) {
              TIMED(c_w2f, mbar_wait(&w2_full[s2], ph2));
              tc_fence_after_sync();
              const uint64_t db = umma_desc_k_sw128(sW2_u + s2 * W2_SLOT);
              if (elect_one()) {
#pragma unroll
                for (int k = 0; k < BK / 16; ++k)
                  umma_bf16_ss_pair(tmem_u + h * (2 * W2_ROWS), da + 2 * k, db + 2 * k, idesc2, (j | (uint32_t)kb | (uint32_t)k) ? 1u : 0u);
                umma_commit_pair(&w2_empty[s2]);
              }
              __syncwarp();
              if (++s2 == W2_SLOTS) { s2 = 0; ph2 ^= 1u; }
            }
          }
          if (elect_one()) {
            umma_commit_pair(hc_empty);
            if (j == (uint32_t)nch - 1) umma_commit_pair(y_full);
          }
          __syncwarp();
        }
        if (GECCO_DBG_ON(p.dbg) && lane == 0) {
          long long* d = p.dbg + (long long)blockIdx.x * 32;
          d[4] = clock64() - t_start; d[5] = c_w1f; d[6] = c_af; d[7] = c_hr; d[8] = c_ye; d[9] = c_w2f; d[21] = c_hf;
        }
      }
    } else if (warp == 3 && lane == 0) {
      // ------------------------------------------------------------ residual loader
      if (p.e.has_res && !(p.e.skip & 2)) {
        uint32_t cnt[EPI_GROUPS] = {0, 0};
        uint32_t it = 0;
        for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
          const int m0 = pb * 2 * BM + (int)rank * BM;
          // every group starts a row block on its dedicated buffer: the first chunk of each group is loaded ahead of the
          // epilogue; the second buffers alias the hidden chunk, which the second GEMM reads until Y is complete
          epi_load_residual_chunk(es, &tma_res, m0, 0, 0, cnt[0], l2_policy(0));
          epi_load_residual_chunk(es, &tma_res, m0, EPI_CHUNK, 1, cnt[1], l2_policy(0));
          mbar_wait(y_full, it & 1u);
          for (int c = 2; c < C / EPI_CHUNK; ++c) epi_load_residual_chunk(es, &tma_res, m0, c * EPI_CHUNK, c & 1, cnt[c & 1], l2_policy(0));
        }
      }
    }
  } else {
    setmaxnreg_inc<232>();
    // ------------------------------------------------------------ activation + final epilogue (each CTA: its 128 rows)
    const int ew = warp - 4;                 // 0..7
    const int q = warp & 3;                  // TMEM lane quadrant of this warp
    const int half = ew >> 2;                // which 64 of the chunk's 128 hidden columns (= k-block of the hidden chunk)
    const EpiThread et = epi_thread_init(es, ew >> 2, threadIdx.x & (EPI_THREADS - 1));
    const uint32_t row = q * 32 + lane;      // row inside the CTA's 128
    const uint32_t h_row = smem_u32(sH) + half * H_KB_BYTES + row * 128u;
    const uint32_t x7 = (row & 7u) << 4;
    const uint32_t tmem_h = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + Y_COLS + half * 64;
    uint32_t g = 0, it = 0, cnt = 0;
    long long c_hf = 0, c_hce = 0, c_yf = 0, c_epi = 0, c_ld = 0, c_act = 0;
    const long long t_start = clock64();
    for (int pb = pair; pb < p.num_pair_blocks; pb += num_pairs, ++it) {
      const int m0 = pb * 2 * BM + (int)rank * BM;
      const float* b1 = p.b1 + (long long)(m0 / p.e.rows_per_cloud) * p.b1_stride + half * 64;
      for (int j = 0; j < nch; ++j, ++g) {
        TIMED(c_hf, mbar_wait(h_full, g & 1u));
        tc_fence_after_sync();
        long long tl0 = 0;
        if (GECCO_DBG_ON(p.dbg)) tl0 = clock64();
        uint32_t r0[32], r1[32];
        tmem_ld32_issue(tmem_h, r0);
        tmem_ld32_issue(tmem_h + 32, r1);
        tmem_ld32_wait(r0);
        tmem_ld32_wait(r1);
        // H(g) is in registers: hand the TMEM buffer back so the first GEMM of the next chunk runs under the activation
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(h_free);
        if (GECCO_DBG_ON(p.dbg)) c_ld += clock64() - tl0;
        const float4* bp = reinterpret_cast<const float4*>(b1 + j * HC);
        uint32_t pk[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 bi = __ldg(bp + i);
          pk[2 * i] = pack_bf16x2(gauss_act(__uint_as_float(r0[4 * i + 0]) + bi.x, p.act_k),
                                  gauss_act(__uint_as_float(r0[4 * i + 1]) + bi.y, p.act_k));
          pk[2 * i + 1] = pack_bf16x2(gauss_act(__uint_as_float(r0[4 * i + 2]) + bi.z, p.act_k),
                                      gauss_act(__uint_as_float(r0[4 * i + 3]) + bi.w, p.act_k));
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float4 bi = __ldg(bp + 8 + i);
          pk[16 + 2 * i] = pack_bf16x2(gauss_act(__uint_as_float(r1[4 * i + 0]) + bi.x, p.act_k),
                                       gauss_act(__uint_as_float(r1[4 * i + 1]) + bi.y, p.act_k));
          pk[16 + 2 * i + 1] = pack_bf16x2(gauss_act(__uint_as_float(r1[4 * i + 2]) + bi.z, p.act_k),
                                           gauss_act(__uint_as_float(r1[4 * i + 3]) + bi.w, p.act_k));
        }
        if (GECCO_DBG_ON(p.dbg)) c_act += clock64() - tl0;
        // the second GEMM of the previous chunk has finished reading the shared-memory chunk
        TIMED(c_hce, mbar_wait(hc_empty, (g & 1u) ^ 1u));
#pragma unroll
        for (int i = 0; i < 8; ++i)
          sts128u(h_row + ((((uint32_t)i) << 4) ^ x7), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        fence_proxy_async_smem();   // generic-proxy writes -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive_leader(h_ready);
      }
      // final epilogue of the row block: Y (+ b2, + residual, statistics) -> x (fp32), xb (bf16)
      epi_prefetch(p.e, et, m0, 0);
      TIMED(c_yf, mbar_wait(y_full, it & 1u));
      tc_fence_after_sync();
      long long t_epi = 0;
      if (GECCO_DBG_ON(p.dbg)) t_epi = clock64();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
      epi_panel<kStats>(p.e, es, et, &tma_o32, &tma_o16, taddr, m0, 0, cnt);
      __syncwarp();
      epi_prefetch(p.e, et, m0, EPI_PANEL);
      epi_panel<kStats>(p.e, es, et, &tma_o32, &tma_o16, taddr + EPI_PANEL, m0, EPI_PANEL, cnt);
      tc_fence_before_sync();
      if (lane == 0) tma_store_wait_read<0>();  // the staging areas (= hidden chunk buffer, W2 ring) are free again
      __syncwarp();
      if (lane == 0) {
        mbar_arrive_leader(y_empty);
        mbar_arrive(epi_done);
      }
      named_bar_sync(1, EPI_GROUPS * EPI_THREADS);
      if (GECCO_DBG_ON(p.dbg)) c_epi += clock64() - t_epi;
    }
    if (GECCO_DBG_ON(p.dbg) && lane == 0 && ew == 0) {
      long long* d = p.dbg + (long long)blockIdx.x * 32;
      d[10] = clock64() - t_start; d[11] = c_hf; d[12] = c_hce; d[13] = c_yf; d[14] = c_epi; d[25] = c_ld; d[26] = c_act;
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

static bool mlp_fused_supported(const gecco_mlp_args& a) {
  return a.c == C && a.hidden >= HC && a.hidden % HC == 0 && a.m > 0 && a.m % (2 * BM) == 0 &&
         a.rows_per_cloud % (2 * BM) == 0 && sm_count() >= 2;
}

static int launch_mlp_fused(const gecco_mlp_args& a, cudaStream_t stream) {
  GECCO_REQUIRE(a.a && a.w1 && a.w2 && a.b1 && a.b2, "mlp: null operand");
  GECCO_REQUIRE(a.res && a.out_f32, "mlp: the fp32 residual stream (res, out_f32) is required");
  GECCO_REQUIRE(mlp_fused_supported(a),
                "mlp: fused kernel needs c == 384, hidden %% 128 == 0, m %% 256 == 0 and rows_per_cloud %% 256 == 0 "
                "(c=%d hidden=%d m=%d rows_per_cloud=%d)", a.c, a.hidden, a.m, a.rows_per_cloud);
  GECCO_REQUIRE(a.valid_rows > 0 && a.valid_rows <= a.rows_per_cloud, "mlp: valid_rows out of range");
  GECCO_REQUIRE(a.act_alpha != 0.f, "mlp: act_alpha must be non-zero");

  const int clouds = ceil_div(a.m, a.rows_per_cloud);
  const uint64_t w1_rows = a.w1_rows_per_cloud ? (uint64_t)a.w1_rows_per_cloud * (clouds - 1) + a.hidden : (uint64_t)a.hidden;
  CUtensorMap ta, tw1, tw2, tres, t32, t16;
  if (int rc = make_tmap_bf16(&ta, a.a, C, a.m, a.lda, BM)) return rc;
  if (int rc = make_tmap_bf16(&tw1, a.w1, C, w1_rows, a.ldw1, HC / 2)) return rc;
  if (int rc = make_tmap_bf16(&tw2, a.w2, a.hidden, C, a.ldw2, W2_ROWS)) return rc;
  if (int rc = make_residual_tmap(a.res, a.ldr, a.m, C, ta, &tres)) return rc;
  if (int rc = make_output_tmaps(a.out_f32, a.ldo32, a.out_bf16, a.ldo16, a.m, C, ta, &t32, &t16)) return rc;

  MParams p;
  p.e.M = a.m; p.e.n_out = C;
  p.e.rows_per_cloud = a.rows_per_cloud; p.e.valid_rows = a.valid_rows;
  p.e.bias = a.b2; p.e.bias_stride = 0;
  p.e.act = 0; p.e.act_k = 0.f;
  p.e.has_res = 1;
  p.e.o32 = a.out_f32;
  p.e.o16 = static_cast<__nv_bfloat16*>(a.out_bf16);
  p.e.stats = a.stats;
  p.e.geom = nullptr; p.e.sigma = nullptr; p.e.sigma_stride = 0; p.e.sigma_data = 1.f; p.e.wx = nullptr;
  p.b1 = a.b1; p.b1_stride = a.b1_stride;
  p.act_k = static_cast<float>(-1.4426950408889634 / (2.0 * (double)a.act_alpha * (double)a.act_alpha));
  p.w1_rows_per_cloud = a.w1_rows_per_cloud;
  p.num_chunks = a.hidden / HC;
  p.num_pair_blocks = a.m / (2 * BM);
  p.dbg = g_gemm_debug;
  p.e.dbg = g_gemm_debug;
  p.e.skip = epi_skip_option();
  p.e.hints = 0;

  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(mlp_fused_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(mlp_fused_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(mlp_fused_kernel)");
    attr_set = true;
  }
  int pairs = sm_count() / 2;
  if (pairs > p.num_pair_blocks) pairs = p.num_pair_blocks;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le = a.stats ? cudaLaunchKernelEx(&cfg, mlp_fused_kernel<true>, ta, tw1, tw2, tres, t32, t16, p)
                           : cudaLaunchKernelEx(&cfg, mlp_fused_kernel<false>, ta, tw1, tw2, tres, t32, t16, p);
  if (le != cudaSuccess) return fail_cuda(le, "mlp_fused_kernel launch");
  GECCO_CHECK_LAUNCH("mlp_fused_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco

extern "C" int gecco_mlp(const gecco_mlp_args* args, void* stream) {
  GECCO_REQUIRE(args != nullptr, "gecco_mlp: null args");
  if (args->anorm.stats != nullptr) return gecco::launch_mlp_pair(*args, static_cast<cudaStream_t>(stream));
  return gecco::launch_mlp_fused(*args, static_cast<cudaStream_t>(stream));
}
