// Pool attention core on the 5th-generation tensor cores (tcgen05 / TMEM), models/set_transformer.py:47-65:
// AttentionPool's scaled_dot_product_attention of the 64 learned inducer queries over the N points of a cloud,
//     o_h[i, :] = sum_n softmax_n(q_h[i] . k_h[n]) v_h[n, :]          (8 heads of 48 channels, q pre-scaled by d^-1/2 log2 e)
// between kv_proj (the tcgen05 GEMM that wrote k | v) and out_proj.
//
// Work item = (cloud, head pair, key split); a CTA runs two items at a time, one per softmax warpgroup, each streaming
// over its 128-point tiles ("units"):
//   * A = [Q_h ; Q_h+1]  (128 stacked (head, inducer) rows x 48, K-major; the warpgroup stages the pair of its item).
//   * S_a = A K_h^T, S_b = A K_h+1^T : 2 x three M128 N128 K16 MMAs into TMEM; rows 0-63 of S_a and rows 64-127 of S_b
//     are the scores of the pair (the other halves are unused cross terms -- the tensor pipe has 10x headroom here, the
//     kernel is bound by streaming k and v from HBM).  K_h tiles arrive by TMA as [128 points x 64 columns] windows
//     starting at column 48h of k.
//   * one thread per stacked row: running max / sum over the tiles (flash-attention recurrence, base-2 exponentials),
//     P = exp2(S - m) written as bf16 into two swizzled K-major k-blocks (points contiguous).
//   * O = P [V_h | V_h+1] : eight M128 N96 K16 MMAs with the pair's v columns as the MN-major B operand, i.e. exactly the
//     [point][channel] boxes TMA delivers (no transpose anywhere; the second 64-channel atom is the next box, LBO);
//     rows of head h use columns 0-47 of O, rows of head h+1 columns 48-95; O lands in TMEM columns S occupied.
//     The thread rescales its 48 fp32 accumulators in registers: acc = acc * 2^(m_old - m_new) + O.
//   * end of an item: the normalised bf16 row ("b h i d -> b i (h d)") when the item covers all keys, else the
//     (acc, m, l) partial for pool_combine_kernel.
// TMEM: warpgroup w owns columns [256 w, 256 w + 256): S_a / O_a at +0, S_b / O_b at +128.
// Shared memory: Q 2 x 16 KB | K window ring 4 x 16 KB | V window ring 4 x 16 KB | P 2 x 32 KB.  K windows are released
// as soon as the first product has read them, V windows only after the second: separate rings keep the early K release
// from queueing behind the V windows, so the next unit's K is in flight while the current one is in its softmax.
//
//   warp 0 : TMA producer          warp 2 : TMEM allocator
//   warp 1 : MMA issuer            warps 4-7 / 8-11 : softmax warpgroups 0 / 1
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace gecco {
namespace {

constexpr int TM = 128;            // points per unit
constexpr int NI = 64;             // inducers
constexpr int HD = 48;             // head dim
constexpr int NH = 8;              // heads
constexpr int NP = NH / 2;         // head pairs
constexpr int C = NH * HD;         // 384
constexpr int SLOTS = 4;           // K window ring, V window ring (two windows per unit each)
constexpr int WIN_BYTES = TM * 128;        // 16 KiB: 128 points x 64 columns (48 used)
constexpr int Q_BYTES = 2 * NI * 128;      // 16 KiB: the 128 stacked rows x 128 B of one head pair
constexpr int P_BYTES = 2 * TM * 128;      // 32 KiB: two k-blocks (64 points each) of 128 rows x 128 B
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 128 + 256;
constexpr int SMEM_BYTES = 1024 /*align*/ + 2 * Q_BYTES + 2 * SLOTS * WIN_BYTES + 2 * P_BYTES + 256 /*barriers*/;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

// kind::f16 instruction descriptor with B MN-major (bit 16): bf16 x bf16 -> fp32.
__host__ __device__ constexpr uint32_t umma_idesc_bf16_bmn(int M, int N) { return umma_idesc_bf16(M, N) | (1u << 16); }
// MN-major, 128B-swizzled B operand spanning two 64-element atoms `lbo_bytes` apart (8-row K groups 1024 B apart).
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t saddr, uint32_t lbo_bytes) {
  uint64_t d = 0;
  d |= static_cast<uint64_t>((saddr & 0x3FFFFu) >> 4);
  d |= static_cast<uint64_t>(lbo_bytes >> 4) << 16;
  d |= static_cast<uint64_t>(1024 >> 4) << 32;
  d |= static_cast<uint64_t>(1) << 46;
  d |= static_cast<uint64_t>(2) << 61;
  return d;
}

struct PParams {
  const __nv_bfloat16* q_ind;  // [8][64][48], pre-scaled
  int clouds, rows_per_cloud, valid_rows;
  int tiles, splits, tps;      // 128-point tiles per cloud, key splits, tiles per split
  int items;                   // clouds * NP * splits
  float* partial;              // [cloud][head][split][64][HD + 2] (splits > 1)
  __nv_bfloat16* out;          // [clouds * 64, ldo] (splits == 1)
  long long ldo;
};

// The units of one warpgroup slot, in the order every role walks them.
struct Cursor {
  int item, item_stride, items;  // current item, stride (2 * gridDim.x), total
  int tile, tile_end;
  int cloud, pair, split;
  __device__ __forceinline__ void open(const PParams& p) {
    if (item >= items) return;
    split = item % p.splits;
    pair = (item / p.splits) % NP;
    cloud = item / (p.splits * NP);
    tile = split * p.tps;
    tile_end = min(p.tiles, tile + p.tps);
  }
  __device__ __forceinline__ void init(const PParams& p, int first, int stride) {
    item = first; item_stride = stride; items = p.items;
    open(p);
  }
  __device__ __forceinline__ bool done() const { return item >= items; }
  __device__ __forceinline__ bool last_of_item() const { return tile + 1 >= tile_end; }
  __device__ __forceinline__ bool first_of_item(const PParams& p) const { return tile == split * p.tps; }
  __device__ __forceinline__ void next(const PParams& p) {
    if (++tile >= tile_end) {
      item += item_stride;
      open(p);
    }
  }
};

__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void tmem_ld32(uint32_t addr, uint32_t (&r)[32]) {
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
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

__global__ void __launch_bounds__(THREADS, 1)
pool_tc_kernel(const __grid_constant__ CUtensorMap tma_k, const __grid_constant__ CUtensorMap tma_v, const PParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                    // [2] stacked query pair of the warpgroup's item
  uint8_t* sK = sQ + 2 * Q_BYTES;        // [SLOTS] K windows
  uint8_t* sV = sK + SLOTS * WIN_BYTES;  // [SLOTS] V windows
  uint8_t* sP = sV + SLOTS * WIN_BYTES;  // [2] probabilities of the two warpgroups
  uint64_t* bars = reinterpret_cast<uint64_t*>(sP + 2 * P_BYTES);
  uint64_t* k_full = bars;               // [SLOTS]
  uint64_t* k_empty = k_full + SLOTS;    // [SLOTS] the first product has read the window
  uint64_t* v_full = k_empty + SLOTS;    // [SLOTS]
  uint64_t* v_empty = v_full + SLOTS;    // [SLOTS] the second product has read the window
  uint64_t* q_ready = v_empty + SLOTS;   // [2] the warpgroup staged the queries of its item: 4 warp arrivals
  uint64_t* s_full = q_ready + 2;        // [2] S of the warpgroup's unit is in TMEM
  uint64_t* p_full = s_full + 2;         // [2] P written and S pulled out of TMEM: 4 warp arrivals
  uint64_t* o_full = p_full + 2;         // [2] the second product is complete
  uint64_t* o_read = o_full + 2;         // [2] O pulled out of TMEM (the region is free): 4 warp arrivals
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_read + 2);

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_k);
    tma_prefetch_desc(&tma_v);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < SLOTS; ++i) {
      mbar_init(&k_full[i], 1);
      mbar_init(&k_empty[i], 1);
      mbar_init(&v_full[i], 1);
      mbar_init(&v_empty[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&q_ready[i], 4);
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&o_full[i], 1);
      mbar_init(&o_read[i], 4);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch_dependents();

  Cursor cur[2];
  cur[0].init(p, blockIdx.x * 2 + 0, gridDim.x * 2);
  cur[1].init(p, blockIdx.x * 2 + 1, gridDim.x * 2);

  if (warp == 0 && lane == 0) {
    // ------------------------------------------------------------ TMA producer: per round K_h, K_h+1 of both warpgroups'
    // units, then their V_h, V_h+1
    uint32_t gk = 0, gv = 0;  // K / V windows issued
    while (!cur[0].done() || !cur[1].done()) {
#pragma unroll
      for (int kind = 0; kind < 2; ++kind) {
#pragma unroll
        for (int w = 0; w < 2; ++w) {
          if (cur[w].done()) continue;
          const int row = cur[w].cloud * p.rows_per_cloud + cur[w].tile * TM;
          for (int j = 0; j < 2; ++j) {
            // K: the window of head 2 pair + j; V: the two 64-column boxes of the pair's 96 channels.  Columns past 384
            // are zero-filled.
            const int col = kind == 0 ? (2 * cur[w].pair + j) * HD : cur[w].pair * 2 * HD + j * 64;
            if (kind == 0) {
              const uint32_t slot = gk % SLOTS, use = gk / SLOTS;
              mbar_wait(&k_empty[slot], (use & 1u) ^ 1u);
              mbar_arrive_expect_tx(&k_full[slot], WIN_BYTES);
              tma_load_2d(sK + slot * WIN_BYTES, &tma_k, &k_full[slot], col, row);
              ++gk;
            } else {
              const uint32_t slot = gv % SLOTS, use = gv / SLOTS;
              mbar_wait(&v_empty[slot], (use & 1u) ^ 1u);
              mbar_arrive_expect_tx(&v_full[slot], WIN_BYTES);
              tma_load_2d(sV + slot * WIN_BYTES, &tma_v, &v_full[slot], col, row);
              ++gv;
            }
          }
        }
      }
#pragma unroll
      for (int w = 0; w < 2; ++w)
        if (!cur[w].done()) cur[w].next(p);
    }
  } else if (uwarp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp, one elected lane issues)
    constexpr uint32_t idesc_s = umma_idesc_bf16(TM, TM);          // M = 128 stacked rows, N = 128 points
    constexpr uint32_t idesc_o = umma_idesc_bf16_bmn(TM, 2 * HD);  // M = 128 stacked rows, N = 96 channels (MN-major V)
    const uint32_t sQ_u = uniform_u32(smem_u32(sQ)), sK_u = uniform_u32(smem_u32(sK)), sV_u = uniform_u32(smem_u32(sV));
    const uint32_t sP_u = uniform_u32(smem_u32(sP));
    const uint32_t tmem_u = uniform_u32(tmem_base);
    uint32_t gk = 0, gv = 0;      // K / V windows consumed (ring positions; both advance in the producer's order)
    uint32_t nS[2] = {0, 0};      // units whose first product has been issued, per warpgroup
    uint32_t nO[2] = {0, 0};      // units whose second product has been issued
    uint32_t nQ[2] = {0, 0};      // items started
    int pend[2] = {0, 0};         // a second product is pending for the warpgroup
    // first product of the warpgroup's next unit
    auto issue_s = [&](int w) {
      // the TMEM region is free once O of the previous unit has been pulled out
      if (nS[w] > 0) mbar_wait(&o_read[w], (nS[w] - 1) & 1u);
      if (cur[w].first_of_item(p)) {
        mbar_wait(&q_ready[w], nQ[w] & 1u);
        ++nQ[w];
      }
      const uint32_t k0 = gk % SLOTS, k1 = (gk + 1) % SLOTS;
      mbar_wait(&k_full[k0], (gk / SLOTS) & 1u);
      mbar_wait(&k_full[k1], ((gk + 1) / SLOTS) & 1u);
      tc_fence_after_sync();
      if (elect_one()) {
        const uint32_t qa = sQ_u + w * Q_BYTES;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          const uint32_t kb = sK_u + (hh ? k1 : k0) * WIN_BYTES;
#pragma unroll
          for (int kk = 0; kk < HD / 16; ++kk)
            umma_bf16_ss(tmem_u + w * 256 + hh * 128, umma_desc_k_sw128(qa) + 2 * kk, umma_desc_k_sw128(kb) + 2 * kk, idesc_s,
                         kk ? 1u : 0u);
        }
        umma_commit(&k_empty[k0]);
        umma_commit(&k_empty[k1]);
        umma_commit(&s_full[w]);
      }
      __syncwarp();
      gk += 2;
      ++nS[w];
      pend[w] = 1;
      cur[w].next(p);
    };
    // second product of the warpgroup's pending unit (V windows are consumed in the order the first products were issued)
    auto issue_o = [&](int w) {
      mbar_wait(&p_full[w], nO[w] & 1u);
      const uint32_t v0 = gv % SLOTS, v1 = (gv + 1) % SLOTS;
      mbar_wait(&v_full[v0], (gv / SLOTS) & 1u);
      mbar_wait(&v_full[v1], ((gv + 1) / SLOTS) & 1u);
      tc_fence_after_sync();
      if (elect_one()) {
        // one product for both heads: N = the pair's 96 channels (two adjacent 64-channel boxes, the second atom one
        // window further: LBO); rows of head h use columns 0-47 of O, rows of head h+1 columns 48-95
        const uint32_t vb = sV_u + v0 * WIN_BYTES;
#pragma unroll
        for (int kk = 0; kk < TM / 16; ++kk) {
          // A: P, K-major, k-block kk / 4 (64 points), 16-point slice kk % 4.  B: V boxes, MN-major: 16 points = 2048 B.
          const uint64_t da = umma_desc_k_sw128(sP_u + w * P_BYTES + (kk >> 2) * (TM * 128)) + 2 * (kk & 3);
          const uint64_t db = umma_desc_mn_sw128(vb + kk * 2048, WIN_BYTES);
          umma_bf16_ss(tmem_u + w * 256, da, db, idesc_o, kk ? 1u : 0u);
        }
        umma_commit(&v_empty[v0]);
        umma_commit(&v_empty[v1]);
        umma_commit(&o_full[w]);
      }
      __syncwarp();
      gv += 2;
      ++nO[w];
      pend[w] = 0;
    };
#pragma unroll
    for (int w = 0; w < 2; ++w)
      if (!cur[w].done()) issue_s(w);
    while (pend[0] || pend[1]) {
#pragma unroll
      for (int w = 0; w < 2; ++w)
        if (pend[w]) issue_o(w);
#pragma unroll
      for (int w = 0; w < 2; ++w)
        if (!cur[w].done()) issue_s(w);
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ softmax warpgroups: one thread per stacked row
    const int w = (warp - 4) >> 2;
    const int q = warp & 3;                       // TMEM lane quadrant
    const uint32_t row = q * 32 + lane;           // stacked row: head 2 pair + (row >> 6), inducer row & 63
    const uint32_t x7 = (row & 7u) << 4;
    const uint32_t t_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + w * 256 + (q >> 1) * 128;
    const uint32_t o_addr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + w * 256 + (q >> 1) * HD;  // this row's O
    const uint32_t p_row = smem_u32(sP) + w * P_BYTES + row * 128u;
    Cursor& c = cur[w];
    uint32_t n = 0;  // units processed
    float m = -INFINITY, l = 0.f;
    float acc[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) acc[d] = 0.f;

    while (!c.done()) {
      if (c.first_of_item(p)) {
        // the queries of this item's head pair (weights) -> swizzled K-major rows of 128 B.  Every first product of the
        // previous item has completed (its s_full was consumed above).
        const int t = threadIdx.x - 128 - w * 128;
        for (int i = t; i < 2 * NI * (HD / 8); i += 128) {
          const int r = i / (HD / 8), ch = i - r * (HD / 8);
          const uint4 v = __ldg(reinterpret_cast<const uint4*>(p.q_ind + ((long long)c.pair * 2 * NI + r) * HD + ch * 8));
          *reinterpret_cast<uint4*>(sQ + w * Q_BYTES + r * 128 + ((ch ^ (r & 7)) << 4)) = v;
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&q_ready[w]);
      }
      const int nvalid = p.valid_rows - c.tile * TM;  // points of this tile that exist (>= 1)
      mbar_wait(&s_full[w], n & 1u);
      tc_fence_after_sync();
      // Reference exponent of this unit.  The first unit of an item takes the row maximum in a pass of its own; later
      // units keep the reference reached so far (any reference gives the same softmax; TMEM is read once instead of
      // twice) and move it afterwards if the unit raised the maximum.
      float mref = m;
      if (c.first_of_item(p)) {
        float mx = -INFINITY;
#pragma unroll 1
        for (int cb = 0; cb < TM; cb += 32) {
          uint32_t s[32];
          tmem_ld32(t_addr + cb, s);
          tmem_ld_wait();
          if (nvalid >= cb + 32) {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, __uint_as_float(s[i]));
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) mx = fmaxf(mx, cb + i < nvalid ? __uint_as_float(s[i]) : -INFINITY);
          }
        }
        mref = mx;
        m = mx;
      }
      // P = 2^(S - mref), bf16, into the swizzled K-major k-blocks; the unit's own maximum on the side
      float sum, umax;
      for (;;) {
        sum = 0.f;
        umax = -INFINITY;
#pragma unroll 1
        for (int cb = 0; cb < TM; cb += 32) {
          uint32_t s[32];
          tmem_ld32(t_addr + cb, s);
          tmem_ld_wait();
          uint32_t pk[16];
          if (nvalid >= cb + 32) {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const float s0 = __uint_as_float(s[2 * i]), s1 = __uint_as_float(s[2 * i + 1]);
              umax = fmaxf(umax, fmaxf(s0, s1));
              const float a = ex2f(s0 - mref), b = ex2f(s1 - mref);
              sum += a + b;
              pk[i] = pack_bf16x2(a, b);
            }
          } else {
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const bool v0 = cb + 2 * i < nvalid, v1 = cb + 2 * i + 1 < nvalid;
              const float s0 = v0 ? __uint_as_float(s[2 * i]) : -INFINITY, s1 = v1 ? __uint_as_float(s[2 * i + 1]) : -INFINITY;
              umax = fmaxf(umax, fmaxf(s0, s1));
              const float a = ex2f(s0 - mref), b = ex2f(s1 - mref);  // 2^-inf = 0
              sum += a + b;
              pk[i] = pack_bf16x2(a, b);
            }
          }
          const uint32_t kb_row = p_row + (cb >> 6) * (TM * 128);  // k-block of 64 points
          const uint32_t ch0 = (cb & 32) >> 3;                     // first 16 B chunk of these 32 points
#pragma unroll
          for (int i = 0; i < 4; ++i)
            sts128(kb_row + (((ch0 + i) << 4) ^ x7), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        }
        // a jump of the maximum by more than 2^64 would overflow the exponentials: redo the unit (warp-uniform, the
        // TMEM loads are collective) with the reference moved first
        if (!__any_sync(0xffffffffu, umax > mref + 64.f)) break;
        if (umax > mref) {
          const float r = ex2f(mref - umax);
          l *= r;
#pragma unroll
          for (int d = 0; d < HD; ++d) acc[d] *= r;
          mref = umax;
          m = umax;
        }
      }
      l += sum;
      fence_proxy_async_smem();
      tc_fence_before_sync();
      __syncwarp();
      if (lane == 0) mbar_arrive(&p_full[w]);
      // O of this unit (same reference as acc)
      mbar_wait(&o_full[w], n & 1u);
      tc_fence_after_sync();
      {
        uint32_t o[HD];
        tmem_ld16(o_addr, o);
        tmem_ld16(o_addr + 16, o + 16);
        tmem_ld16(o_addr + 32, o + 32);
        tmem_ld_wait();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&o_read[w]);
#pragma unroll
        for (int d = 0; d < HD; ++d) acc[d] += __uint_as_float(o[d]);
      }
      if (umax > m) {  // move the reference for the following units
        const float r = ex2f(m - umax);
        l *= r;
#pragma unroll
        for (int d = 0; d < HD; ++d) acc[d] *= r;
        m = umax;
      }
      ++n;
      if (c.last_of_item()) {
        const int head = 2 * c.pair + (row >> 6), ind = row & 63;
        if (p.splits == 1) {
          const float inv = 1.0f / l;
          uint4* dst = reinterpret_cast<uint4*>(p.out + ((long long)c.cloud * NI + ind) * p.ldo + head * HD);
#pragma unroll
          for (int i = 0; i < HD / 8; ++i)
            dst[i] = make_uint4(pack_bf16x2(acc[8 * i + 0] * inv, acc[8 * i + 1] * inv), pack_bf16x2(acc[8 * i + 2] * inv, acc[8 * i + 3] * inv),
                                pack_bf16x2(acc[8 * i + 4] * inv, acc[8 * i + 5] * inv), pack_bf16x2(acc[8 * i + 6] * inv, acc[8 * i + 7] * inv));
        } else {
          float* dst = p.partial + ((((long long)c.cloud * NH + head) * p.splits + c.split) * NI + ind) * (HD + 2);
#pragma unroll
          for (int d = 0; d < HD; d += 2) *reinterpret_cast<float2*>(dst + d) = make_float2(acc[d], acc[d + 1]);
          *reinterpret_cast<float2*>(dst + HD) = make_float2(m, l);
        }
        m = -INFINITY;
        l = 0.f;
#pragma unroll
        for (int d = 0; d < HD; ++d) acc[d] = 0.f;
      }
      c.next(p);
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

bool pool_tc_supported(const gecco_pool_args& a) {
  return a.heads == NH && a.head_dim == HD && a.inducers == NI && a.rows_per_cloud % TM == 0 && a.ld % 8 == 0 &&
         a.k_off % 8 == 0 && a.v_off % 8 == 0 && a.ldo % 8 == 0 && a.valid_rows >= 1 && a.valid_rows <= a.rows_per_cloud &&
         (reinterpret_cast<uintptr_t>(a.kv) & 15) == 0 && (reinterpret_cast<uintptr_t>(a.out_bf16) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(a.q_inducers) & 15) == 0;
}

// `combine` is set when the result was left as key-split partials for pool_combine_kernel; *splits_used is their count.
int launch_pool_tc(const gecco_pool_args& a, cudaStream_t stream, int* splits_used) {
  GECCO_REQUIRE(pool_tc_supported(a), "pool attention (tcgen05): unsupported shape");
  const __nv_bfloat16* kv = static_cast<const __nv_bfloat16*>(a.kv);
  const long long rows = (long long)a.clouds * a.rows_per_cloud;
  CUtensorMap tk, tv;
  if (int rc = make_tmap_bf16(&tk, kv + a.k_off, C, rows, a.ld, TM)) return rc;
  if (int rc = make_tmap_bf16(&tv, kv + a.v_off, C, rows, a.ld, TM)) return rc;

  PParams p;
  p.q_ind = static_cast<const __nv_bfloat16*>(a.q_inducers);
  p.clouds = a.clouds; p.rows_per_cloud = a.rows_per_cloud; p.valid_rows = a.valid_rows;
  p.tiles = ceil_div(a.valid_rows, TM);
  const int sms = sm_count();
  // key splits: enough (cloud, pair, split) items for the 2 x SMs warpgroup slots, bounded by the caller's partial buffer
  int splits = (2 * sms) / (a.clouds * NP);
  if (splits > a.splits) splits = a.splits;
  if (splits > p.tiles) splits = p.tiles;
  if (splits < 1 || a.partial == nullptr) splits = 1;
  p.tps = ceil_div(p.tiles, splits);
  p.splits = ceil_div(p.tiles, p.tps);
  p.items = a.clouds * NP * p.splits;
  p.partial = a.partial;
  p.out = static_cast<__nv_bfloat16*>(a.out_bf16);
  p.ldo = a.ldo;
  *splits_used = p.splits;
  int grid = ceil_div(p.items, 2);
  if (grid > sms) grid = sms;

  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(pool_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(pool_tc_kernel)");
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
  cudaError_t le = cudaLaunchKernelEx(&cfg, pool_tc_kernel, tk, tv, p);
  if (le != cudaSuccess) return fail_cuda(le, "pool_tc_kernel launch");
  GECCO_CHECK_LAUNCH("pool_tc_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco
