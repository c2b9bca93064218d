// Row-tile epilogue shared by the tcgen05 kernels: drains a 128-row x 192-column fp32 accumulator panel from
// TMEM in 32-column chunks and applies, in this order,
//   + bias[cloud][n]  + xyz embed  -> activation -> + residual -> AdaGN statistics -> fp32 / bf16 stores.
// The statistics are per (cloud, group of W consecutive columns), W a compile-time parameter that divides the panel
// (EpiStats below).
// The TMEM layout gives every thread one ROW of the tile; global memory wants whole row segments per request, so all
// global traffic of the epilogue goes through TMA and swizzled shared memory.
// Two epilogue groups of 128 threads (4 warps each, warp q <-> TMEM lanes 32q..) work on alternate chunks.  Each group
// owns "X" buffers of 128 rows x 32 fp32 columns (16 KB, SWIZZLE_128B): the loader thread TMA-loads the fp32 residual
// chunk into one, every thread adds its accumulator row IN PLACE, and each warp bulk-stores its 32 x 32 block straight
// from the same buffer (res_full / res_empty mbarriers).  With a residual a group has two X buffers, so the residual
// of chunk i+1 is in flight while chunk i is processed and chunk i-1's store drains; without a residual one buffer
// serves as plain output staging.  The bf16 copy goes through a per-warp 2 KB staging area (SWIZZLE_64B).
#pragma once
#include "common.cuh"
#include "ptx.cuh"

#include <type_traits>

namespace gecco {

constexpr int EPI_THREADS = 128;                      // per group
constexpr int EPI_GROUPS = 2;
constexpr int EPI_CHUNK = 32;                         // columns per chunk
constexpr int EPI_PANEL = 192;                        // columns per panel (16 AdaGN groups of 12 at C = 384)
constexpr int EPI_RES_BYTES = 128 * EPI_CHUNK * 4;    // one fp32 chunk (TMA box {32, 128}, SWIZZLE_128B): an X buffer
constexpr int EPI_O16_BYTES = 128 * EPI_CHUNK * 2;    // one bf16 chunk (TMA box {32, 128}, SWIZZLE_64B)
constexpr int EPI_BIAS_BYTES = 8 * 384;                // per-warp bias staging (3 chunks x 32 floats)
constexpr int EPI_NUM_BARS = 4 * EPI_GROUPS;          // res_full[group][2] | res_empty[group][2]

struct EpiParams {
  int M, n_out;
  int rows_per_cloud, valid_rows;
  const float* bias;  // [clouds][bias_stride] or nullptr
  int bias_stride;
  int act;      // GECCO_ACT_*: the kernel's ACT template parameter applies it; at ACT == GECCO_ACT_GAUSSIAN, 0 means none
  float act_k;  // -log2(e) / (2 alpha^2) (the Gaussians)
  int has_res;
  float* o32;           // fp32 output or nullptr (written through its tensor map)
  __nv_bfloat16* o16;   // bf16 output or nullptr
  double* stats;  // [clouds][n_out / W][2] or nullptr (W: the statistics width the kernel was instantiated for)
  const float* geom;  // [clouds, valid_rows, 3] or nullptr
  const float* sigma;
  int sigma_stride;
  float sigma_data;
  const float* wx;  // [n_out, 3]
  int skip;         // development aid (gecco_set_option("epi_skip")): 1 no output stores, 2 no residual, 4 no proxy fence, 8 no statistics atomics
  long long* dbg;   // development aid: [grid][32] cycle counters, slots 16..21 (nullptr in production)
  int hints;        // L2 residency hints (ptx.cuh l2_policy kinds): bits 2-3 residual loads, 4-5 fp32 stores, 6-7 bf16 stores
};

struct EpiSmem {
  uint8_t* x0;   // [group] x EPI_RES_BYTES, 1024 B aligned: X buffer 0 of every group
  uint8_t* x1;   // [group] x EPI_RES_BYTES: X buffer 1 (only with a residual)
  uint8_t* o16;  // [group][warp] x 2 KB bf16 staging (32 rows x 64 B, 64 B swizzle)
  uint8_t* bias; // [group][warp] x 384 B
  uint64_t* res_full;   // [group][2], count 1 + tx
  uint64_t* res_empty;  // [group][2], count 4 (one arrival per warp of the group)
};

// Shared memory the epilogue needs for a given output configuration (1024 B aligned pieces), and its carving.
__host__ __device__ inline int epi_smem_bytes(bool has_res, bool has_o32, bool has_o16) {
  return (has_res ? 2 : (has_o32 ? 1 : 0)) * EPI_GROUPS * EPI_RES_BYTES + (has_o16 ? EPI_GROUPS * EPI_O16_BYTES : 0) +
         EPI_BIAS_BYTES;
}
// Returns the first byte after the epilogue's area.
__device__ __forceinline__ uint8_t* epi_smem_carve(EpiSmem& es, uint8_t* base, bool has_res, bool has_o32, bool has_o16) {
  es.x0 = base;
  if (has_res || has_o32) base += EPI_GROUPS * EPI_RES_BYTES;
  es.x1 = base;
  if (has_res) base += EPI_GROUPS * EPI_RES_BYTES;
  es.o16 = base;
  if (has_o16) base += EPI_GROUPS * EPI_O16_BYTES;
  es.bias = base;
  return base + EPI_BIAS_BYTES;
}
// One thread, before the block-wide (or cluster-wide) barrier that publishes the mbarriers.
__device__ __forceinline__ void epi_bar_init(const EpiSmem& es) {
  for (int i = 0; i < 2 * EPI_GROUPS; ++i) {
    mbar_init(&es.res_full[i], 1);
    mbar_init(&es.res_empty[i], EPI_THREADS / 32);
  }
}

// Loader side (one thread): the residual chunk at column col0 for group g; cnt = chunks loaded for that group so far.
__device__ __forceinline__ void epi_load_residual_chunk(const EpiSmem& sm, const CUtensorMap* tma_res, int m0, int col0,
                                                        int g, uint32_t& cnt, uint64_t pol) {
  const uint32_t b = cnt & 1u, phase = (cnt >> 1) & 1u;
  mbar_wait(&sm.res_empty[g * 2 + b], phase ^ 1u);
  mbar_arrive_expect_tx(&sm.res_full[g * 2 + b], EPI_RES_BYTES);
  tma_load_2d_h((b ? sm.x1 : sm.x0) + g * EPI_RES_BYTES, tma_res, &sm.res_full[g * 2 + b], col0, m0, pol);
  ++cnt;
}
// The residual chunks of one panel in the order the epilogue consumes them (chunk c belongs to group c & 1).
__device__ __forceinline__ void epi_load_residual_panel(const EpiParams& p, const EpiSmem& sm, const CUtensorMap* tma_res,
                                                        int m0, int n0, uint32_t (&cnt)[EPI_GROUPS]) {
  const uint64_t pol = l2_policy((p.hints >> 2) & 3);
#pragma unroll 1
  for (int c = 0; c < EPI_PANEL / EPI_CHUNK; ++c) {
    const int col0 = n0 + c * EPI_CHUNK;
    if (col0 >= p.n_out) break;
    epi_load_residual_chunk(sm, tma_res, m0, col0, c & 1, cnt[c & 1], pol);
  }
}

// Sum over the 32 lanes of v[OFF + (lane % N)] lands in lane (N a power of two <= 32): log2(N) halving steps
// (N - 1 shuffles; 31 instead of 32 x 5 at N = 32), then 5 - log2(N) butterfly steps over the lanes holding the same slot.
template <int N, int OFF, int S>
__device__ __forceinline__ float warp_reduce_scatter(float (&v)[S], int lane) {
  static_assert(N >= 1 && N <= 32 && (N & (N - 1)) == 0 && OFF + N <= S, "reduce-scatter width");
#pragma unroll
  for (int off = N / 2; off >= 1; off >>= 1) {
    const bool upper = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = upper ? v[OFF + i] : v[OFF + i + off];
      const float keep = upper ? v[OFF + i + off] : v[OFF + i];
      v[OFF + i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  float r = v[OFF];
#pragma unroll
  for (int off = N; off < 32; off <<= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
  return r;
}

// Register layout of the AdaGN statistics a thread accumulates for its row over one panel, at a group width of W
// columns (W = 0: no statistics).  Each thread sees three of the panel's six chunks (2 k + grp, k = 0..2).
//  - W divides the chunk (4, 8, 16, 32): only the groups of those three chunks, slot 2 (k (32 / W) + j / W) + moment for
//    column j of its k-th chunk;
//  - W = 12, 24 (groups straddle chunks): every group of the panel, slot 2 g + moment (the other chunks' slots stay 0).
// The warp reduce-scatters the slots in rounds of at most 32 (the last one padded to a power of two: kRegs registers)
// and one lane per slot adds it into stats[cloud][n_out / W][{sum, sumsq}].
constexpr int epi_pow2_ceil(int x) { return x <= 1 ? 1 : 2 * epi_pow2_ceil((x + 1) / 2); }
template <int W>
struct EpiStats {
  static_assert(W == 0 || (W > 0 && EPI_PANEL % W == 0 && W % 4 == 0), "statistics width must divide the panel");
  static constexpr bool kLocal = W > 0 && EPI_CHUNK % W == 0;
  static constexpr int kSlots = W == 0 ? 0 : kLocal ? 3 * 2 * (EPI_CHUNK / W) : 2 * (EPI_PANEL / W);
  static constexpr int kRounds = (kSlots + 31) / 32;
  // lanes reduce-scatter round r spans (slots 32 r ...)
  static constexpr __host__ __device__ int width(int r) { return kSlots - 32 * r >= 32 ? 32 : epi_pow2_ceil(kSlots - 32 * r); }
  static constexpr int kRegs = W == 0 ? 1 : 32 * (kRounds - 1) + width(kRounds - 1);
  // slot of column j of panel chunk c (c = 2 k + grp)
  static constexpr __host__ __device__ int slot(int c, int j) {
    return kLocal ? 2 * ((c >> 1) * (EPI_CHUNK / W) + j / W) : 2 * ((c * EPI_CHUNK + j) / W);
  }
};

__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t addr, float a, float b, float c, float d) {
  asm volatile("st.shared.v4.f32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void sts128u(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// The hidden projection's activation (include/gecco_b200.h GECCO_ACT_*) on accumulator + bias v, a compile-time choice of
// each kernel instantiation; k = -log2(e) / (2 alpha^2).
template <int ACT>
__device__ __forceinline__ float epi_act(float v, float k) {
  static_assert(ACT == GECCO_ACT_GAUSSIAN || ACT == GECCO_ACT_GAUSSIAN_RAW || ACT == GECCO_ACT_RELU, "activation code");
  if constexpr (ACT == GECCO_ACT_GAUSSIAN) return fmaf(ex2_approx(v * v * k), 1.0f / 0.28f, -0.7f / 0.28f);
  else if constexpr (ACT == GECCO_ACT_GAUSSIAN_RAW) return ex2_approx(v * v * k);
  else return fmaxf(v, 0.f);
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread.
__device__ __forceinline__ void tmem_ld32_issue(uint32_t addr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,"
      "%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(addr)
      : "memory");
}
// tcgen05.wait::ld with the loaded registers as operands, so that no use of them can be scheduled above the wait.
__device__ __forceinline__ void tmem_ld32_wait(uint32_t (&r)[32]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

// Per-thread constants of the epilogue (shared-window addresses of the staging areas), computed once per kernel.
struct EpiThread {
  int grp, q, lane;
  uint32_t x7;          // (lane & 7) << 4: 128 B swizzle term of row `lane` (and of tile row q*32+lane)
  uint32_t xw0;         // X buffer 0, this thread's row (q*32+lane of the group's 128): piece j at  xw | ((j << 4) ^ x7)
  uint32_t xs0;         // X buffer 0, this warp's 32 rows (source of the fp32 bulk store)
  uint32_t xdelta;      // X buffer 1 = X buffer 0 + xdelta (multiple of 1024 B)
  uint32_t x3, w16;     // bf16 staging, write side: piece j of row `lane` at  w16 | ((j << 4) ^ x3)
  uint32_t s16;         // base of this warp's bf16 staging area (source of the bf16 bulk store)
  uint32_t bias;        // per-warp bias staging: 3 chunks x 32 floats
};

__device__ __forceinline__ EpiThread epi_thread_init(const EpiSmem& sm, int grp, int tid) {
  EpiThread t;
  // q and the warp-level staging bases are warp-uniform: say so (shuffle), the bulk-store operands then live in uniform
  // registers instead of being broadcast lane by lane in front of every store
  t.grp = grp; t.q = __shfl_sync(0xffffffffu, tid >> 5, 0); t.lane = tid & 31;
  const uint32_t lane = t.lane, w = grp * 4 + t.q;
  t.x7 = (lane & 7u) << 4;
  t.xs0 = smem_u32(sm.x0) + grp * EPI_RES_BYTES + t.q * 4096u;
  t.xw0 = t.xs0 + lane * 128u;
  t.xdelta = smem_u32(sm.x1) - smem_u32(sm.x0);
  t.x3 = ((lane >> 1) & 3u) << 4;
  const uint32_t s16 = smem_u32(sm.o16) + w * 2048u;
  t.w16 = s16 + lane * 64u;
  t.s16 = s16;
  t.bias = smem_u32(sm.bias) + w * 384u;
  return t;
}

// Bias of this group's three chunks of panel (m0, n0): loaded into registers one panel AHEAD (the global-load latency
// overlaps the whole previous panel), staged into the warp's shared-memory area right before the panel is drained.
struct EpiBias { float b[3]; };
__device__ __forceinline__ void epi_bias_load(const EpiParams& p, const EpiThread& t, int m0, int n0, EpiBias& r) {
  r.b[0] = r.b[1] = r.b[2] = 0.f;
  if (p.bias == nullptr) return;
  const int cloud = (m0 + t.q * 32) / p.rows_per_cloud;
  const float* bp = p.bias + (long long)cloud * p.bias_stride + n0 + t.grp * EPI_CHUNK + t.lane;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int col = n0 + (2 * k + t.grp) * EPI_CHUNK + t.lane;
    if (col < p.n_out) r.b[k] = __ldg(bp + 2 * k * EPI_CHUNK);
  }
}
__device__ __forceinline__ void epi_bias_stage(const EpiParams& p, const EpiThread& t, const EpiBias& r) {
  if (p.bias == nullptr) return;
#pragma unroll
  for (int k = 0; k < 3; ++k)
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(t.bias + k * 128u + t.lane * 4u), "f"(r.b[k]) : "memory");
  __syncwarp();
}
// Load + stage in one go (kernels that cannot look one panel ahead).
__device__ __forceinline__ void epi_prefetch(const EpiParams& p, const EpiThread& t, int m0, int n0) {
  EpiBias r;
  epi_bias_load(p, t, m0, n0, r);
  epi_bias_stage(p, t, r);
}

#define EPI_TIMED(slot, stmt)                                                        \
  do {                                                                              \
    if (GECCO_DBG_ON(p.dbg)) {                                                         \
      const long long t0__ = clock64();                                             \
      stmt;                                                                         \
      if (t.lane == 0 && t.q == 0 && t.grp == 0) p.dbg[(long long)blockIdx.x * 32 + (slot)] += clock64() - t0__; \
    } else {                                                                        \
      stmt;                                                                         \
    }                                                                               \
  } while (0)

// One 32-column chunk after its accumulator values (+ bias) are in registers.  C: chunk index inside the panel
// (compile-time, so the AdaGN group of every column is static).  W: statistics width (0: none).  ACT: the activation;
// the Gaussian instantiation applies it when p.act != 0, the others always.
template <int W, int C, int ACT = GECCO_ACT_GAUSSIAN>
__device__ __forceinline__ void epi_chunk(const EpiParams& p, const EpiSmem& sm, const EpiThread& t, float (&v)[EPI_CHUNK],
                                          int m0, int col0, bool rows_valid, bool row_valid, float g0, float g1, float g2,
                                          const CUtensorMap* tma_o32, const CUtensorMap* tma_o16,
                                          float (&st)[EpiStats<W>::kRegs], uint32_t& cnt) {
  if (p.geom != nullptr) {
    const float4* wp = reinterpret_cast<const float4*>(p.wx + (long long)col0 * 3);
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) {
      if (col0 + 4 * j < p.n_out) {
        const float4 w0 = __ldg(wp + 3 * j), w1 = __ldg(wp + 3 * j + 1), w2 = __ldg(wp + 3 * j + 2);
        v[4 * j + 0] += g0 * w0.x + g1 * w0.y + g2 * w0.z;
        v[4 * j + 1] += g0 * w0.w + g1 * w1.x + g2 * w1.y;
        v[4 * j + 2] += g0 * w1.z + g1 * w1.w + g2 * w2.x;
        v[4 * j + 3] += g0 * w2.y + g1 * w2.z + g2 * w2.w;
      }
    }
  }
  if (ACT != GECCO_ACT_GAUSSIAN || p.act) {
#pragma unroll
    for (int j = 0; j < EPI_CHUNK; ++j) v[j] = epi_act<ACT>(v[j], p.act_k);
  }
  // The previous chunk's bulk stores have finished reading their staging (its X buffer and the bf16 area): with a
  // residual that X buffer goes back to the loader, which refills it while this chunk is processed.
  const bool use_res = p.has_res && !(p.skip & 2);
  const uint32_t b = use_res ? (cnt & 1u) : 0u;
  const uint32_t xw = t.xw0 + b * t.xdelta, xs = t.xs0 + b * t.xdelta;
  EPI_TIMED(18, { if (t.lane == 0) tma_store_wait_read<0>(); __syncwarp(); });
  if (use_res) {
    if (t.lane == 0 && cnt > 0) mbar_arrive(&sm.res_empty[t.grp * 2 + (b ^ 1u)]);
    EPI_TIMED(17, mbar_wait(&sm.res_full[t.grp * 2 + b], (cnt >> 1) & 1u));
#pragma unroll
    for (int h = 0; h < 2; ++h) {  // two batches of four loads: latency overlapped, bounded register use
      float4 x[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) x[j] = lds128(xw | (((4 * h + j) << 4) ^ t.x7));
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[16 * h + 4 * j + 0] += x[j].x; v[16 * h + 4 * j + 1] += x[j].y;
        v[16 * h + 4 * j + 2] += x[j].z; v[16 * h + 4 * j + 3] += x[j].w;
      }
    }
  }
  if (!rows_valid && !row_valid) {
#pragma unroll
    for (int j = 0; j < EPI_CHUNK; ++j) v[j] = 0.f;  // padding rows stay exactly zero
  }
  if constexpr (W != 0) {
#pragma unroll
    for (int j = 0; j < EPI_CHUNK; ++j) {
      const int sl = EpiStats<W>::slot(C, j);  // static: n0 is a multiple of 192
      st[sl] += v[j];
      st[sl + 1] = fmaf(v[j], v[j], st[sl + 1]);
    }
  }
  // this thread's row goes back into the X buffer (over its own residual values), the warp's 32 x 32 block is then
  // bulk-stored from there: one tensor store per output (box {32 columns, 32 rows}; rows / columns outside the
  // matrix are clipped by the tensor map)
  long long tf0__ = 0;
  if (GECCO_DBG_ON(p.dbg)) tf0__ = clock64();
  if (p.o32 != nullptr) {
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) sts128(xw | ((j << 4) ^ t.x7), v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
  }
  if (p.o16 != nullptr) {
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 8; ++j)
      sts128u(t.w16 | ((j << 4) ^ t.x3), pack_bf16x2(v[8 * j], v[8 * j + 1]), pack_bf16x2(v[8 * j + 2], v[8 * j + 3]),
              pack_bf16x2(v[8 * j + 4], v[8 * j + 5]), pack_bf16x2(v[8 * j + 6], v[8 * j + 7]));
  }
  long long tf1__ = 0, tf2__ = 0;
  if (GECCO_DBG_ON(p.dbg)) tf1__ = clock64();
  if (!(p.skip & 4)) fence_proxy_async_smem();
  __syncwarp();
  if (GECCO_DBG_ON(p.dbg)) tf2__ = clock64();
  if (elect_one() && !(p.skip & 1)) {  // lane 0 (the bulk groups are per thread: the same lane waits for them)
    if (p.o32 != nullptr) tma_store_2d_addr_h(tma_o32, xs, col0, m0 + t.q * 32, l2_policy((p.hints >> 4) & 3));
    if (p.o16 != nullptr) tma_store_2d_addr_h(tma_o16, t.s16, col0, m0 + t.q * 32, l2_policy((p.hints >> 6) & 3));
    tma_store_commit();
  }
  if (GECCO_DBG_ON(p.dbg) && t.lane == 0 && t.q == 0 && t.grp == 0) {
    const long long tf3__ = clock64();
    p.dbg[(long long)blockIdx.x * 32 + 19] += tf1__ - tf0__;
    p.dbg[(long long)blockIdx.x * 32 + 29] += tf2__ - tf1__;
    p.dbg[(long long)blockIdx.x * 32 + 30] += tf3__ - tf2__;
  }
  ++cnt;
}

// Epilogue side (all threads of both groups).  taddr: TMEM address of (lane quadrant q, panel column 0).
// `cnt` counts the chunks this group has processed (the loader keeps the same count per group).  The bias of (m0, n0)
// must have been staged by this thread (epi_bias_stage / epi_prefetch).  The group's three chunks (grp, grp + 2, grp + 4) are software
// pipelined: the TMEM load of the next chunk is issued as soon as the current one has been consumed, because
// tcgen05.ld latency is several hundred cycles while the tensor core is streaming accumulators through TMEM.
template <int W, int ACT = GECCO_ACT_GAUSSIAN>
__device__ __forceinline__ void epi_panel(const EpiParams& p, const EpiSmem& sm, const EpiThread& t,
                                          const CUtensorMap* tma_o32, const CUtensorMap* tma_o16, uint32_t taddr, int m0,
                                          int n0, uint32_t& cnt) {
  const int row = m0 + t.q * 32 + t.lane;
  const int cloud = (m0 + t.q * 32) / p.rows_per_cloud;  // warp-uniform (rows_per_cloud % 32 == 0)
  const int row_in_cloud = row - cloud * p.rows_per_cloud;
  const bool row_valid = row < p.M && row_in_cloud < p.valid_rows;
  const bool rows_valid = m0 + t.q * 32 + 31 < p.M && (m0 + t.q * 32 + 31 - cloud * p.rows_per_cloud) < p.valid_rows;

  uint32_t rr[2][EPI_CHUNK];
  const uint32_t ta = taddr + t.grp * EPI_CHUNK;
  if (n0 + t.grp * EPI_CHUNK < p.n_out) tmem_ld32_issue(ta, rr[0]);

  float g0 = 0.f, g1 = 0.f, g2 = 0.f;
  if (p.geom != nullptr && row_valid) {
    // geom is compact [clouds, valid_rows, 3]; output rows are padded to rows_per_cloud
    const float s = __ldg(p.sigma + (long long)cloud * p.sigma_stride);
    const float c_in = 1.0f / sqrtf(p.sigma_data * p.sigma_data + s * s);
    const float* gp = p.geom + ((long long)cloud * p.valid_rows + row_in_cloud) * 3;
    g0 = c_in * __ldg(gp + 0);
    g1 = c_in * __ldg(gp + 1);
    g2 = c_in * __ldg(gp + 2);
  }
  using Stats = EpiStats<W>;
  float st[Stats::kRegs];  // {sum, sumsq} of this row per group (layout: EpiStats)
#pragma unroll
  for (int i = 0; i < Stats::kRegs; ++i) st[i] = 0.f;
  auto step = [&](auto kc) {
    constexpr int k = decltype(kc)::value;
    if (n0 + (2 * k + t.grp) * EPI_CHUNK < p.n_out) {  // uniform over the epilogue group
      float4 b[EPI_CHUNK / 4];
      if (p.bias != nullptr) {
#pragma unroll
        for (int j = 0; j < EPI_CHUNK / 4; ++j) b[j] = lds128(t.bias + k * 128u + j * 16u);
      } else {
#pragma unroll
        for (int j = 0; j < EPI_CHUNK / 4; ++j) b[j] = make_float4(0.f, 0.f, 0.f, 0.f);
      }
      EPI_TIMED(16, tmem_ld32_wait(rr[k & 1]));
      float v[EPI_CHUNK];
#pragma unroll
      for (int j = 0; j < EPI_CHUNK / 4; ++j) {
        v[4 * j + 0] = __uint_as_float(rr[k & 1][4 * j + 0]) + b[j].x;
        v[4 * j + 1] = __uint_as_float(rr[k & 1][4 * j + 1]) + b[j].y;
        v[4 * j + 2] = __uint_as_float(rr[k & 1][4 * j + 2]) + b[j].z;
        v[4 * j + 3] = __uint_as_float(rr[k & 1][4 * j + 3]) + b[j].w;
      }
      if (k < 2 && n0 + (2 * k + 2 + t.grp) * EPI_CHUNK < p.n_out) tmem_ld32_issue(ta + (2 * k + 2) * EPI_CHUNK, rr[(k + 1) & 1]);
      const int col0 = n0 + (2 * k + t.grp) * EPI_CHUNK;
      if constexpr (W != 0) {  // the AdaGN group of every column must be static: one instantiation per chunk index
        if (t.grp == 0)
          epi_chunk<W, 2 * k, ACT>(p, sm, t, v, m0, col0, rows_valid, row_valid, g0, g1, g2, tma_o32, tma_o16, st, cnt);
        else
          epi_chunk<W, 2 * k + 1, ACT>(p, sm, t, v, m0, col0, rows_valid, row_valid, g0, g1, g2, tma_o32, tma_o16, st, cnt);
      } else {
        epi_chunk<0, 0, ACT>(p, sm, t, v, m0, col0, rows_valid, row_valid, g0, g1, g2, tma_o32, tma_o16, st, cnt);
      }
    }
  };
  step(std::integral_constant<int, 0>{});
  step(std::integral_constant<int, 1>{});
  step(std::integral_constant<int, 2>{});
  if constexpr (W != 0) {
    long long ts0__ = 0;
    if (GECCO_DBG_ON(p.dbg)) ts0__ = clock64();
    auto round = [&](auto kr) {
      constexpr int r = decltype(kr)::value;
      constexpr int N = Stats::width(r);
      const float mine = warp_reduce_scatter<N, 32 * r>(st, t.lane);
      const int s = 32 * r + (N == 32 ? t.lane : (t.lane & (N - 1)));  // this lane's slot
      // [group][{sum, sumsq}] of the cloud
      const int gidx = Stats::kLocal ? (n0 / W) * 2 + (2 * (s / (64 / W)) + t.grp) * (64 / W) + s % (64 / W)
                                     : (n0 / W) * 2 + s;
      const bool own = (N == 32 && 32 * r + 32 <= Stats::kSlots) || (t.lane < N && s < Stats::kSlots);
      if (own && gidx < (p.n_out / W) * 2 && m0 + t.q * 32 < p.M)
        if (!(p.skip & 8)) atomicAdd(p.stats + (long long)cloud * (p.n_out / W) * 2 + gidx, static_cast<double>(mine));
    };
    round(std::integral_constant<int, 0>{});
    if constexpr (Stats::kRounds > 1) round(std::integral_constant<int, 1>{});
    static_assert(Stats::kRounds <= 2, "at most two reduce-scatter rounds");
    if (GECCO_DBG_ON(p.dbg) && t.lane == 0 && t.q == 0 && t.grp == 0) p.dbg[(long long)blockIdx.x * 32 + 20] += clock64() - ts0__;
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Fast path for the bf16-only projections (k|v|q, MLP up): bias (+ activation ACT, GECCO_ACT_NONE: none) -> bf16, whole tiles only (all
// 128 rows valid, n_out a multiple of the panel), no residual / statistics / fp32 copy / xyz embed.  Everything is
// compile-time, the three chunks of a warp are drained from TMEM back to back (three tcgen05.ld in flight) and the
// accumulator slot is handed back to the MMA issuer BEFORE the conversion and the stores; the three 32 x 32 bf16 blocks
// go through three staging areas per warp and leave with one fence and one bulk group.
// Staging areas per warp (2 KB each).  3: one fence and one bulk group per tile; 1: the three blocks go out one after the
// other through the same area (wait for the previous store to have read it).  The epilogue warps idle more than half of
// the time behind the MMA issuer once the accumulator is released early, so the single area is the default: the 32 KB it
// frees go to the weight ring, which is what the issuer actually waits for.
#ifndef GECCO_EPI_FAST_BUFS
#define GECCO_EPI_FAST_BUFS 1
#endif
constexpr int EPI_FAST_BUFS = GECCO_EPI_FAST_BUFS;
constexpr int EPI_FAST_O16_BYTES = EPI_FAST_BUFS * EPI_O16_BYTES;  // per group: 4 warps x EPI_FAST_BUFS x 2 KB

__host__ __device__ inline int epi_fast_smem_bytes() { return EPI_GROUPS * EPI_FAST_O16_BYTES + EPI_BIAS_BYTES; }

template <int ACT, typename ReleaseFn>
__device__ __forceinline__ void epi_tile_fast(const EpiParams& p, const EpiThread& t, const CUtensorMap* tma_o16, uint32_t taddr,
                                              int m0, int n0, uint32_t stage_base, bool row_valid, ReleaseFn release) {
  uint32_t rr[3][EPI_CHUNK];
  const uint32_t ta = taddr + t.grp * EPI_CHUNK;
#pragma unroll
  for (int k = 0; k < 3; ++k) tmem_ld32_issue(ta + 2 * k * EPI_CHUNK, rr[k]);
  const bool zero_row = p.valid_rows < p.rows_per_cloud && !row_valid;  // padding rows are written as exact zeros
  const uint32_t wst = stage_base + (uint32_t)(t.grp * 4 + t.q) * (EPI_FAST_BUFS * 2048u);  // this warp: 32 rows x 64 B, 64 B swizzle
  if (EPI_FAST_BUFS == 3 && t.lane == 0) tma_store_wait_read<0>();  // the previous tile's stores have read the staging areas
  uint32_t pk[EPI_FAST_BUFS == 3 ? 3 : 1][EPI_CHUNK / 2];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    uint32_t (&pw)[EPI_CHUNK / 2] = pk[EPI_FAST_BUFS == 3 ? k : 0];
    float4 b[EPI_CHUNK / 4];
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) b[j] = lds128(t.bias + k * 128u + j * 16u);
    tmem_ld32_wait(rr[k]);
    if (k == 0) release();  // tcgen05.wait::ld covers all three loads: the accumulator slot goes back to the MMA issuer
#pragma unroll
    for (int j = 0; j < EPI_CHUNK / 4; ++j) {
      float v0 = __uint_as_float(rr[k][4 * j + 0]) + b[j].x, v1 = __uint_as_float(rr[k][4 * j + 1]) + b[j].y;
      float v2 = __uint_as_float(rr[k][4 * j + 2]) + b[j].z, v3 = __uint_as_float(rr[k][4 * j + 3]) + b[j].w;
      if constexpr (ACT != GECCO_ACT_NONE) {
        v0 = epi_act<ACT>(v0, p.act_k);
        v1 = epi_act<ACT>(v1, p.act_k);
        v2 = epi_act<ACT>(v2, p.act_k);
        v3 = epi_act<ACT>(v3, p.act_k);
      }
      pw[2 * j] = zero_row ? 0u : pack_bf16x2(v0, v1);
      pw[2 * j + 1] = zero_row ? 0u : pack_bf16x2(v2, v3);
    }
    if (EPI_FAST_BUFS != 3) {
      // single staging area: the previous block's store has read it; stage, fence, store this block
      if (t.lane == 0) tma_store_wait_read<0>();
      __syncwarp();
#pragma unroll
      for (int j = 0; j < EPI_CHUNK / 8; ++j)
        sts128u((wst + t.lane * 64u) | ((j << 4) ^ t.x3), pw[4 * j], pw[4 * j + 1], pw[4 * j + 2], pw[4 * j + 3]);
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        tma_store_2d_addr_h(tma_o16, wst, n0 + (2 * k + t.grp) * EPI_CHUNK, m0 + t.q * 32, l2_policy((p.hints >> 6) & 3));
        tma_store_commit();
      }
    }
  }
  if (EPI_FAST_BUFS == 3) {
    __syncwarp();  // lane 0's wait on the previous stores covers the whole warp's staging areas
#pragma unroll
    for (int k = 0; k < 3; ++k)
#pragma unroll
      for (int j = 0; j < EPI_CHUNK / 8; ++j)
        sts128u((wst + k * 2048u + t.lane * 64u) | ((j << 4) ^ t.x3), pk[EPI_FAST_BUFS == 3 ? k : 0][4 * j], pk[EPI_FAST_BUFS == 3 ? k : 0][4 * j + 1],
                pk[EPI_FAST_BUFS == 3 ? k : 0][4 * j + 2], pk[EPI_FAST_BUFS == 3 ? k : 0][4 * j + 3]);
    fence_proxy_async_smem();
    __syncwarp();
    if (elect_one()) {
#pragma unroll
      for (int k = 0; k < 3; ++k) tma_store_2d_addr(tma_o16, wst + k * 2048u, n0 + (2 * k + t.grp) * EPI_CHUNK, m0 + t.q * 32);
      tma_store_commit();
    }
  }
}

}  // namespace gecco
