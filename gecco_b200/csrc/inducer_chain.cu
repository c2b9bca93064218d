// The inducer side of Broadcast.forward (models/set_transformer.py:106-112) as ONE kernel per layer:
//     pooled = combine(key-split partials of AttentionPool)             (:61-63, when the pool core split the keys)
//     h  = out_proj(pooled)                                             (:64)
//     h  = norm_1(h, t)            AdaGN, statistics over (64 inducers, 12 channels)   (:108)
//     h  = mlp(h)                  Linear -> GaussianActivation -> Linear               (:109)
//     h  = norm_2(h, t)                                                                 (:110)
//     k | v = in_proj[C:3C](h)     key / value projection of unpool = nn.MultiheadAttention (:112), + V^T for the core
// Round 1 / 2 ran this as eight launches (combine, 4 GEMMs, 2 AdaGN applies, V transpose) of 6-10 us each on 32-128
// CTAs: 0.4 % of the FLOPs and 10 % of the step.  Here a CLUSTER of four CTAs owns two clouds (128 rows = one
// tcgen05 M tile): every CTA computes a quarter of the output columns of every stage (so it streams a quarter of each
// weight matrix from L2), the 64 x 12 AdaGN groups of its columns are local to its accumulator, and the stages are
// separated by cluster barriers.  Activations travel between the stages as bf16 through global memory (L2): 48-96 KB per
// stage and cluster.
//
//   warp 0 : TMA producer (weights of the NEXT stage are prefetched before the cluster barrier, the A operand after it)
//   warp 1 : MMA issuer (M=128, N=96 / 192, one TMEM accumulator)
//   warp 2 : TMEM allocator      warp 3 : -
//   warps 4-19 : combine, then the epilogues: thread = (row, quarter of the CTA's columns)
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace gecco {
extern long long* g_gemm_debug;  // gemm_pair.cu: optional debug buffer (gecco_set_debug_buffer)
namespace {

constexpr int TM = 128;           // rows per cluster: two clouds x 64 inducers
constexpr int NI = 64;
constexpr int C = 384;
constexpr int HID = 768;
constexpr int NH = 8, HD = 48;
constexpr int GS = 12;            // AdaGN group width (32 groups of 12 channels)
constexpr int CL = 4;             // CTAs per cluster
constexpr int BK = 64;
constexpr int A_BYTES = TM * BK * 2;       // 16 KiB
constexpr int W_BYTES = 192 * BK * 2;      // 24 KiB (stages with 96 columns per CTA use half)
constexpr int STAGE_BYTES = A_BYTES + W_BYTES;
constexpr int RING = 4;
constexpr int STG_BYTES = 32 * 96;      // per epilogue warp: 32 rows x 96 B (48 bf16 / 24 fp32), or V^T 48 channels x 64 B
constexpr int THREADS = 128 + 512;
constexpr int EPI_THREADS_ALL = 512;
constexpr int TMEM_COLS = 256;
constexpr int NSTAGES = 4;
constexpr int SMEM_BYTES = 1024 + RING * STAGE_BYTES + 2 * 2 * 2 * 96 * 4 /*AdaGN scale / bias*/ + 2 * 4 * 96 * 4 /*raw AdaGN weights*/ + 480 * 4 /*biases*/ + 16 * 4 * 4 /*reduction*/ + 256 + 16 * STG_BYTES;

struct CParams {
  int clouds, m;                        // m = clouds * 64 rows
  int first_stage;                      // 0: whole chain; 3: only the key / value projection (cached inducer states)
  // pool combine
  const float* partial; int splits;     // [cloud][head][split][64][HD + 2]; splits <= 1: `pooled` is final already
  __nv_bfloat16* pooled;
  // AdaGN norm_1 / norm_2: scale.weight, scale.bias, bias.weight, bias.bias ([C] each), t [clouds]
  const float* n_w[2][4];
  const float* t; int t_stride; float eps;
  // biases
  const float *b_mlp0, *b_mlp2, *b_kv;
  float act_k;                          // -log2(e) / (2 alpha^2)
  // activations
  __nv_bfloat16 *hn, *hh, *h3, *khv, *vt;
  float* cache_out;                     // optional fp32 [m, C]: norm_2 output (the inducer cache of SetTransformer.forward)
  long long* dbg;                       // development aid: [grid][32] globaltimer stamps (gecco_set_debug_buffer), else nullptr
};

__device__ __forceinline__ long long gtime() {
  long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}
#define STAMP(slot)                                                                   \
  do {                                                                                \
    if (p.dbg != nullptr && stamp_thread) p.dbg[(long long)blockIdx.x * 32 + (slot)] = gtime(); \
  } while (0)

__device__ __forceinline__ void cluster_arrive() { asm volatile("barrier.cluster.arrive.release;" ::: "memory"); }
__device__ __forceinline__ void cluster_wait() { asm volatile("barrier.cluster.wait.acquire;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// K of stage s and output columns per CTA
__device__ __forceinline__ int stage_k(int s) { return s == 2 ? HID : C; }
__device__ __forceinline__ int stage_n(int s) { return (s & 1) ? 192 : 96; }

// N (24 or 48) accumulator columns of this thread's row starting at TMEM address taddr
__device__ __forceinline__ void tmem_ld8(uint32_t addr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(addr)
               : "memory");
}
template <int N>
__device__ __forceinline__ void tmem_load(uint32_t taddr, float (&v)[N]) {
  static_assert(N == 24 || N == 48, "24 or 48 columns");
  uint32_t r[N];
  tmem_ld16(taddr, r);
  if (N == 48) {
    tmem_ld16(taddr + 16, r + 16);
    tmem_ld16(taddr + 32, r + 32);
  } else {
    tmem_ld8(taddr + 16, r + 16);
  }
  tmem_ld_wait();
#pragma unroll
  for (int i = 0; i < N; ++i) {
    asm volatile("" : "+r"(r[i]));  // no use of the loaded registers is scheduled above tcgen05.wait::ld
    v[i] = __uint_as_float(r[i]);
  }
}

// Row-per-thread values -> the warp's staging tile (32 rows x ROWB bytes) -> global memory with consecutive lanes on
// consecutive 16-byte pieces of a row (a thread storing its own row would scatter every request over 32 lines).
template <int ROWB>
__device__ __forceinline__ void warp_tile_to_global(const uint8_t* stg, uint8_t* gdst, long long row_stride_bytes, int rows_valid,
                                                    int lane) {
  constexpr int CH = ROWB / 16;
  __syncwarp();
#pragma unroll
  for (int idx = lane; idx < 32 * CH; idx += 32) {
    const int r = idx / CH, ch = idx - r * CH;
    if (r < rows_valid)
      *reinterpret_cast<uint4*>(gdst + r * row_stride_bytes + ch * 16) = *reinterpret_cast<const uint4*>(stg + r * ROWB + ch * 16);
  }
  __syncwarp();
}
template <int N>
__device__ __forceinline__ void stage_bf16(uint8_t* stg_row, const float (&v)[N]) {
#pragma unroll
  for (int j = 0; j < N / 8; ++j) {
    uint4 pk;
    pk.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
    pk.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
    pk.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
    pk.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(stg_row + 16 * j) = pk;
  }
}

template <int N>
__device__ __forceinline__ void store_bf16(__nv_bfloat16* dst, const float (&v)[N]) {
#pragma unroll
  for (int j = 0; j < N / 8; ++j) {
    uint4 pk;
    pk.x = pack_bf16x2(v[8 * j + 0], v[8 * j + 1]);
    pk.y = pack_bf16x2(v[8 * j + 2], v[8 * j + 3]);
    pk.z = pack_bf16x2(v[8 * j + 4], v[8 * j + 5]);
    pk.w = pack_bf16x2(v[8 * j + 6], v[8 * j + 7]);
    *reinterpret_cast<uint4*>(dst + 8 * j) = pk;
  }
}

// kAct: the MLP's hidden activation (GECCO_ACT_GAUSSIAN, GECCO_ACT_GAUSSIAN_RAW or GECCO_ACT_RELU)
template <int kAct>
__global__ void __cluster_dims__(CL, 1, 1) __launch_bounds__(THREADS, 1)
inducer_chain_kernel(const __grid_constant__ CUtensorMap ta0, const __grid_constant__ CUtensorMap ta1,
                     const __grid_constant__ CUtensorMap ta2, const __grid_constant__ CUtensorMap ta3,
                     const __grid_constant__ CUtensorMap tw0, const __grid_constant__ CUtensorMap tw1,
                     const __grid_constant__ CUtensorMap tw2, const __grid_constant__ CUtensorMap tw3, const CParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* ring = smem;
  float* s_norm = reinterpret_cast<float*>(smem + RING * STAGE_BYTES);  // [norm][cloud][{scale, bias}][96]
  float* s_nw = s_norm + 2 * 2 * 2 * 96;                                 // [norm][4][96] raw AdaGN weights of this CTA's columns
  float* s_bias = s_nw + 2 * 4 * 96;                                     // b_mlp0 [192] | b_mlp2 [96] | b_kv [192] of this CTA's columns
  float* s_red = s_bias + 480;                                           // [warp 0..15][4]
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_red + 64);
  uint64_t* full = bars;             // [RING]
  uint64_t* empty = bars + RING;     // [RING]
  uint64_t* acc_full = bars + 2 * RING;
  uint64_t* acc_empty = acc_full + 1;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 1);
  uint8_t* s_stage = reinterpret_cast<uint8_t*>(bars) + 256;  // [16 warps] x STG_BYTES

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int m0 = (blockIdx.x / CL) * TM;

  const CUtensorMap* tas[NSTAGES] = {&ta0, &ta1, &ta2, &ta3};
  const CUtensorMap* tws[NSTAGES] = {&tw0, &tw1, &tw2, &tw3};

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGES; ++s) {
      tma_prefetch_desc(tas[s]);
      tma_prefetch_desc(tws[s]);
    }
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < RING; ++i) {
      mbar_init(&full[i], 1);
      mbar_init(&empty[i], 1);
    }
    mbar_init(acc_full, 1);
    mbar_init(acc_empty, EPI_THREADS_ALL / 32);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // static weights of this CTA's columns -> shared memory, under the tail of the preceding kernel
  if (threadIdx.x >= 128) {
    const int et = threadIdx.x - 128;
    const int rk = (int)cluster_ctarank();
    for (int i = et; i < 480; i += EPI_THREADS_ALL) {
      float b;
      if (i < 192) b = p.b_mlp0 ? __ldg(p.b_mlp0 + rk * 192 + i) : 0.f;
      else if (i < 288) b = p.b_mlp2 ? __ldg(p.b_mlp2 + rk * 96 + i - 192) : 0.f;
      else b = __ldg(p.b_kv + rk * 192 + i - 288);
      s_bias[i] = b;
    }
    if (p.first_stage == 0)
      for (int i = et; i < 2 * 4 * 96; i += EPI_THREADS_ALL) s_nw[i] = __ldg(p.n_w[i / 384][(i / 96) & 3] + rk * 96 + i % 96);
  }
  pdl_wait();
  pdl_launch_dependents();

  const int s_begin = p.first_stage;
  const bool stamp_thread = threadIdx.x == 128 || threadIdx.x == 32;
  if (threadIdx.x == 128) STAMP(0);
  if (uwarp == 0) {
    // ------------------------------------------------------------ TMA producer (whole warp runs the loop, one lane issues)
    int slot = 0;
    uint32_t phase = 0;
    for (int s = s_begin; s < NSTAGES; ++s) {
      const int nkb = stage_k(s) / BK;
      const int wn = stage_n(s);
      const uint32_t bytes = A_BYTES + (uint32_t)wn * BK * 2;
      const int npre = nkb < RING ? nkb : RING;
      // the weights of this stage do not depend on the previous one: in flight across the cluster barrier
      int pslot = slot;
      uint32_t pphase = phase;
      cluster_arrive();
      for (int kb = 0; kb < npre; ++kb) {
        mbar_wait(&empty[pslot], pphase ^ 1u);
        if (lane == 0) {
          mbar_arrive_expect_tx(&full[pslot], bytes);
          tma_load_2d(ring + pslot * STAGE_BYTES + A_BYTES, tws[s], &full[pslot], kb * BK, rank * wn);
        }
        if (++pslot == RING) { pslot = 0; pphase ^= 1u; }
      }
      cluster_wait();          // the previous stage's activations (all four CTAs' columns) are in global memory
      fence_proxy_async_all();
      for (int kb = 0; kb < nkb; ++kb) {
        if (kb >= npre) {
          mbar_wait(&empty[slot], phase ^ 1u);
          if (lane == 0) {
            mbar_arrive_expect_tx(&full[slot], bytes);
            tma_load_2d(ring + slot * STAGE_BYTES + A_BYTES, tws[s], &full[slot], kb * BK, rank * wn);
          }
        }
        if (lane == 0) tma_load_2d(ring + slot * STAGE_BYTES, tas[s], &full[slot], kb * BK, m0);
        if (++slot == RING) { slot = 0; phase ^= 1u; }
      }
    }
  } else if (uwarp == 1) {
    // ------------------------------------------------------------ MMA issuer
    const uint32_t ring_u = uniform_u32(smem_u32(ring));
    const uint32_t tmem_u = uniform_u32(tmem_base);
    int slot = 0;
    uint32_t phase = 0;
    uint32_t it = 0;
    for (int s = s_begin; s < NSTAGES; ++s, ++it) {
      cluster_arrive();
      cluster_wait();
      const int nkb = stage_k(s) / BK;
      const uint32_t idesc = (s & 1) ? umma_idesc_bf16(TM, 192) : umma_idesc_bf16(TM, 96);
      mbar_wait(acc_empty, (it & 1u) ^ 1u);
      tc_fence_after_sync();
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full[slot], phase);
        if (kb == 0) STAMP(20 + s);
        tc_fence_after_sync();
        const uint64_t da = umma_desc_k_sw128(ring_u + slot * STAGE_BYTES);
        const uint64_t db = umma_desc_k_sw128(ring_u + slot * STAGE_BYTES + A_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) umma_bf16_ss(tmem_u, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          umma_commit(&empty[slot]);
        }
        __syncwarp();
        if (++slot == RING) { slot = 0; phase ^= 1u; }
      }
      if (elect_one()) umma_commit(acc_full);
      __syncwarp();
    }
  } else if (warp < 4) {
    for (int s = s_begin; s < NSTAGES; ++s) {
      cluster_arrive();
      cluster_wait();
    }
  } else {
    // ------------------------------------------------------------ combine + epilogues
    const int et = threadIdx.x - 128;      // 0..511
    const int q = warp & 3;                // TMEM lane quadrant
    const int g = (warp - 4) >> 2;         // column quarter of the CTA's accumulator
    const int row = q * 32 + lane;         // row of the cluster tile
    const int lc = row >> 6;               // local cloud
    const uint32_t tlane = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    uint8_t* stg = s_stage + (warp - 4) * STG_BYTES;
    const int rows_valid = min(32, max(0, p.m - (m0 + q * 32)));
    const long long grow0 = (long long)m0 + q * 32;  // first row of this warp

    if (s_begin == 0) {
      named_bar_sync(3, EPI_THREADS_ALL);  // s_nw staged
      // AdaGN scale(t) / bias(t) of this CTA's 96 columns for both norms and both clouds (raw weights staged before the
      // dependency wait)
      for (int i = et; i < 2 * 2 * 96; i += EPI_THREADS_ALL) {
        const int c = i % 96, cl = (i / 96) & 1, n = i / 192;
        const int cloud = m0 / NI + cl;
        const float tc = cloud < p.clouds ? __ldg(p.t + (long long)cloud * p.t_stride) : 0.f;
        const float* nw = s_nw + n * 4 * 96 + c;
        s_norm[((n * 2 + cl) * 2 + 0) * 96 + c] = tc * nw[0] + nw[96];
        s_norm[((n * 2 + cl) * 2 + 1) * 96 + c] = tc * nw[192] + nw[288];
      }
      // pool combine: this CTA merges the key splits of heads 2 rank, 2 rank + 1 of both clouds; half a (cloud, head,
      // inducer) row (24 values) per thread
      if (p.splits > 1) {
        const int r = et >> 1, half = et & 1;
        const int cl = r >> 7, head = 2 * rank + ((r >> 6) & 1), i = r & 63;
        const int cloud = m0 / NI + cl;
        if (cloud < p.clouds) {
          const float* base = p.partial + (((long long)cloud * NH + head) * p.splits) * NI * (HD + 2) + (long long)i * (HD + 2);
          float M = -INFINITY;
          for (int sp = 0; sp < p.splits; ++sp) M = fmaxf(M, __ldg(base + (long long)sp * NI * (HD + 2) + HD));
          float L = 0.f;
          float acc[HD / 2];
#pragma unroll
          for (int d = 0; d < HD / 2; ++d) acc[d] = 0.f;
          for (int sp = 0; sp < p.splits; ++sp) {
            const float2* pr = reinterpret_cast<const float2*>(base + (long long)sp * NI * (HD + 2));
            float2 x[HD / 4];
#pragma unroll
            for (int d = 0; d < HD / 4; ++d) x[d] = __ldg(pr + half * (HD / 4) + d);
            const float2 ml = __ldg(pr + HD / 2);
            const float w = (ml.x == -INFINITY) ? 0.f : ex2f(ml.x - M);
            L += w * ml.y;
#pragma unroll
            for (int d = 0; d < HD / 4; ++d) {
              acc[2 * d] += w * x[d].x;
              acc[2 * d + 1] += w * x[d].y;
            }
          }
          const float inv = 1.0f / L;
#pragma unroll
          for (int d = 0; d < HD / 2; ++d) acc[d] *= inv;
          store_bf16<HD / 2>(p.pooled + ((long long)cloud * NI + i) * C + head * HD + half * (HD / 2), acc);
        }
      }
      fence_proxy_async_all();
    }
    named_bar_sync(3, EPI_THREADS_ALL);  // s_norm visible
    STAMP(1);

    uint32_t it = 0;
    for (int s = s_begin; s < NSTAGES; ++s, ++it) {
      cluster_arrive();
      cluster_wait();
      STAMP(2 + 4 * s);
      mbar_wait(acc_full, it & 1u);
      STAMP(3 + 4 * s);
      tc_fence_after_sync();
      if ((s & 1) == 0) {
        // ---------------- 96 columns per CTA, 24 per thread: (+ bias) -> AdaGN over the (64 rows, 12 columns) groups -> bf16
        const int n = s >> 1;  // norm_1 / norm_2
        float v[24];
        tmem_load<24>(tlane + g * 24, v);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty);
        const int lcol = g * 24;              // first column inside the CTA's 96
        const int col0 = rank * 96 + lcol;    // first output channel of this thread
        if (s == 2) {
          const float4* b4 = reinterpret_cast<const float4*>(s_bias + 192 + lcol);
#pragma unroll
          for (int i = 0; i < 6; ++i) {
            const float4 b = b4[i];
            v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
          }
        }
        float red[4];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          float a = 0.f, b = 0.f;
#pragma unroll
          for (int j = 0; j < GS; ++j) {
            a += v[k * GS + j];
            b = fmaf(v[k * GS + j], v[k * GS + j], b);
          }
          red[k] = a;
          red[2 + k] = b;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) red[k] = warp_sum(red[k]);
        if (lane == 0) {
#pragma unroll
          for (int k = 0; k < 4; ++k) s_red[(warp - 4) * 4 + k] = red[k];
        }
        named_bar_sync(3, EPI_THREADS_ALL);
        const float* r0 = s_red + (warp - 4) * 4;
        const float* r1 = s_red + ((warp - 4) ^ 1) * 4;  // the other 32 rows of this cloud, same columns
        const float* sc = s_norm + ((n * 2 + lc) * 2 + 0) * 96 + lcol;
        const float* bi = sc + 96;
        constexpr float inv_n = 1.0f / (NI * GS);
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          // fixed summation order (lower warp first): both warps of the cloud get bit-identical statistics
          const float* ra = (warp & 1) ? r1 : r0;
          const float* rb = (warp & 1) ? r0 : r1;
          const float mean = (ra[k] + rb[k]) * inv_n;
          float var = fmaf(-mean, mean, (ra[2 + k] + rb[2 + k]) * inv_n);
          var = var < 0.f ? 0.f : var;
          const float rstd = rsqrtf(var + p.eps);
#pragma unroll
          for (int j = 0; j < GS; ++j) {
            const float a = sc[k * GS + j] * rstd;
            v[k * GS + j] = fmaf(a, v[k * GS + j] - mean, bi[k * GS + j]);
          }
        }
        stage_bf16<24>(stg + lane * 48, v);
        warp_tile_to_global<48>(stg, reinterpret_cast<uint8_t*>((s == 0 ? p.hn : p.h3) + grow0 * C + col0), C * 2, rows_valid, lane);
        if (s == 2 && p.cache_out != nullptr) {
#pragma unroll
          for (int j = 0; j < 6; ++j)
            *reinterpret_cast<float4*>(stg + lane * 96 + 16 * j) = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          warp_tile_to_global<96>(stg, reinterpret_cast<uint8_t*>(p.cache_out + grow0 * C + col0), C * 4, rows_valid, lane);
        }
        named_bar_sync(3, EPI_THREADS_ALL);  // s_red may be rewritten by the next AdaGN stage
      } else {
        // ---------------- 192 columns per CTA, 48 per thread: + bias (-> activation) -> bf16
        __nv_bfloat16* out = s == 1 ? p.hh : p.khv;
        float v[48];
        tmem_load<48>(tlane + g * 48, v);
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(acc_empty);
        const int lcol = g * 48;
        const int col0 = rank * 192 + lcol;
        const float4* b4 = reinterpret_cast<const float4*>(s_bias + (s == 1 ? 0 : 288) + lcol);
#pragma unroll
        for (int i = 0; i < 12; ++i) {
          const float4 b = b4[i];
          v[4 * i] += b.x; v[4 * i + 1] += b.y; v[4 * i + 2] += b.z; v[4 * i + 3] += b.w;
        }
        if (s == 1) {
#pragma unroll
          for (int i = 0; i < 48; ++i) {
            if constexpr (kAct == GECCO_ACT_GAUSSIAN) v[i] = fmaf(ex2f(v[i] * v[i] * p.act_k), 1.0f / 0.28f, -0.7f / 0.28f);
            else if constexpr (kAct == GECCO_ACT_GAUSSIAN_RAW) v[i] = ex2f(v[i] * v[i] * p.act_k);
            else v[i] = fmaxf(v[i], 0.f);
          }
        }
        stage_bf16<48>(stg + lane * 96, v);
        warp_tile_to_global<96>(stg, reinterpret_cast<uint8_t*>(out + grow0 * HID + col0), HID * 2, rows_valid, lane);
        if (s == 3 && col0 >= C && p.vt != nullptr) {
          // V^T of the cloud for the unpool core: vt[cloud][c][i].  Staging tile [48 channels][32 inducers]; a global row of
          // the tile is the 64 B  vt[cloud][col0 - C + c][32 (q & 1) .. + 32)
#pragma unroll
          for (int i = 0; i < 48; ++i) *reinterpret_cast<__nv_bfloat16*>(stg + i * 64 + lane * 2) = __float2bfloat16(v[i]);
          __syncwarp();
          if (rows_valid > 0) {
            uint8_t* vt = reinterpret_cast<uint8_t*>(p.vt + ((long long)(m0 / NI + lc) * C + (col0 - C)) * NI + (q & 1) * 32);
#pragma unroll
            for (int idx = lane; idx < 48 * 4; idx += 32) {
              const int c = idx >> 2, ch = idx & 3;
              *reinterpret_cast<uint4*>(vt + (long long)c * NI * 2 + ch * 16) = *reinterpret_cast<const uint4*>(stg + c * 64 + ch * 16);
            }
          }
          __syncwarp();
        }
      }
      STAMP(4 + 4 * s);
      fence_proxy_async_all();  // generic-proxy global writes -> the next stage's TMA reads (after the cluster barrier)
      STAMP(5 + 4 * s);
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

}  // namespace

bool inducer_chain_supported(const gecco_chain_args& a) {
  return a.inducers == NI && a.c == C && a.hidden == HID && a.heads == NH && a.groups == C / GS && a.clouds > 0 &&
         sm_count() >= CL;
}

int launch_inducer_chain(const gecco_chain_args& a, cudaStream_t stream) {
  GECCO_REQUIRE(inducer_chain_supported(a),
                "inducer chain: only 64 inducers, C = 384, hidden = 768, 8 heads, 32 AdaGN groups are supported");
  GECCO_REQUIRE(a.first_stage == 0 || a.first_stage == 3, "inducer chain: first_stage must be 0 or 3");
  GECCO_REQUIRE(a.hn && a.hh && a.h3 && a.khv && a.pooled, "inducer chain: null activation buffer");
  GECCO_REQUIRE(a.w_kv && a.b_kv, "inducer chain: null key / value projection");
  if (a.first_stage == 0) {
    GECCO_REQUIRE(a.w_pool_out && a.w_mlp0 && a.w_mlp2 && a.b_mlp0 && a.b_mlp2 && a.t, "inducer chain: null weight");
    for (int n = 0; n < 2; ++n)
      for (int i = 0; i < 4; ++i) GECCO_REQUIRE(a.norm[n][i] != nullptr, "inducer chain: null AdaGN weight");
    GECCO_REQUIRE(a.splits <= 1 || a.partial != nullptr, "inducer chain: key-split partials missing");
  }
  const int m = a.clouds * NI;
  CUtensorMap ta[4], tw[4];
  const int act = mlp_act_of(a.act);
  GECCO_REQUIRE(act == GECCO_ACT_GAUSSIAN || act == GECCO_ACT_GAUSSIAN_RAW || act == GECCO_ACT_RELU,
                "inducer chain: unknown activation code %d", a.act);
  const void* as[4] = {a.pooled, a.hn, a.hh, a.h3};
  const void* ws[4] = {a.w_pool_out ? a.w_pool_out : a.w_kv, a.w_mlp0 ? a.w_mlp0 : a.w_kv, a.w_mlp2 ? a.w_mlp2 : a.w_kv, a.w_kv};
  const int ks[4] = {C, C, HID, C};
  const int ns[4] = {C, HID, C, HID};
  for (int s = 0; s < 4; ++s) {
    if (int rc = make_tmap_bf16(&ta[s], as[s], ks[s], m, ks[s], TM)) return rc;
    if (a.first_stage == 3 && s < 3) { tw[s] = ta[s]; continue; }
    if (int rc = make_tmap_bf16(&tw[s], ws[s], ks[s], ns[s], ks[s], ns[s] / CL)) return rc;
  }
  if (a.first_stage == 3)
    if (int rc = make_tmap_bf16(&tw[3], ws[3], ks[3], ns[3], ks[3], ns[3] / CL)) return rc;

  CParams p = {};
  p.clouds = a.clouds; p.m = m; p.first_stage = a.first_stage;
  p.partial = a.partial; p.splits = a.splits;
  p.pooled = static_cast<__nv_bfloat16*>(a.pooled);
  for (int n = 0; n < 2; ++n)
    for (int i = 0; i < 4; ++i) p.n_w[n][i] = a.norm[n][i];
  p.t = a.t; p.t_stride = a.t_stride; p.eps = a.eps;
  p.b_mlp0 = a.b_mlp0; p.b_mlp2 = a.b_mlp2; p.b_kv = a.b_kv;
  p.act_k = a.first_stage == 0 ? act_k_of(act, a.act_alpha) : 0.f;
  p.hn = static_cast<__nv_bfloat16*>(a.hn); p.hh = static_cast<__nv_bfloat16*>(a.hh);
  p.h3 = static_cast<__nv_bfloat16*>(a.h3); p.khv = static_cast<__nv_bfloat16*>(a.khv);
  p.vt = static_cast<__nv_bfloat16*>(a.vt);
  p.cache_out = a.cache_out;
  p.dbg = g_gemm_debug;

  using KernelFn = void (*)(CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap, CUtensorMap,
                            CUtensorMap, CParams);
  static const KernelFn kernels[3] = {inducer_chain_kernel<GECCO_ACT_GAUSSIAN>, inducer_chain_kernel<GECCO_ACT_GAUSSIAN_RAW>,
                                      inducer_chain_kernel<GECCO_ACT_RELU>};  // [act - GECCO_ACT_GAUSSIAN]
  static bool attr_set = false;
  if (!attr_set) {
    for (KernelFn k : kernels) {
      cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
      if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(inducer_chain_kernel)");
    }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(CL * ceil_div(m, TM));
  cfg.blockDim = dim3(THREADS);
  cfg.dynamicSmemBytes = SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le = cudaLaunchKernelEx(&cfg, kernels[act - GECCO_ACT_GAUSSIAN], ta[0], ta[1], ta[2], ta[3], tw[0], tw[1], tw[2], tw[3], p);
  if (le != cudaSuccess) return fail_cuda(le, "inducer_chain_kernel launch");
  GECCO_CHECK_LAUNCH("inducer_chain_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco

extern "C" int gecco_inducer_chain(const gecco_chain_args* args, void* stream) {
  if (args == nullptr) {
    gecco::set_error("gecco_inducer_chain: null args");
    return GECCO_ERR_INVALID;
  }
  return gecco::launch_inducer_chain(*args, static_cast<cudaStream_t>(stream));
}
