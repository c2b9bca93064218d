// Unpool attention core on the 5th-generation tensor cores (tcgen05 / TMEM), models/set_transformer.py:90,112:
// nn.MultiheadAttention(query = points, key = value = the 64 inducers of the cloud) between its in- and out-projections,
//     y[r, 48h .. 48h+47] = softmax_i(q_h[r] . k_h[i]) v_h[i]        (8 heads of 48 channels, q pre-scaled by d^-1/2 log2 e)
// One CTA per SM streams over (128-row tile, head) pairs of one or two clouds; nothing is serialised per tile:
//   * K [64 x 384] (six 128B-swizzled k-blocks; B operand of the first product, N = 64 inducers) and V^T [384 x 64]
//     (B operand of the second product: N = 48 channels of head h, K = 64 inducers; produced once per layer by
//     transpose_v_kernel) stay in shared memory for all tiles of a cloud.
//   * Q_h: a [128 x 64] window starting at column 48h (the 16 extra columns are ignored) arrives by TMA in a 4-slot ring.
//   * S_h = Q_h K_h^T: three M128 N64 K16 MMAs into one of two TMEM buffers; two softmax warpgroups (even / odd heads,
//     one thread per row) pull S_h into registers, exponentiate, and write P_h as bf16 into a swizzled k-block;
//     O_h = P_h V_h: four M128 N48 K16 MMAs into TMEM columns 48h.
//   * after signalling P of its next head, a warpgroup drains the finished O of its previous head, normalises by the row
//     sums it kept in registers, stages the [128 x 48] bf16 block and stores it with one bulk tensor store.
// TMEM: O [0, 384) | S buffers [384, 448), [448, 512).
// Shared memory: Q ring 4 x 16 KB, K 48 KB, V^T 48 KB, P 2 x 16 KB, output staging 2 x 12 KB.
//
//   warp 0 : TMA producer (Q per head; K, V^T per cloud)      warp 2 : TMEM allocator
//   warp 1 : MMA issuer (whole warp, one elected lane issues) warps 4-7 / 8-11 : softmax + output of the even / odd heads
#include "common.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

namespace gecco {
namespace {

constexpr int TM = 128;            // rows per tile
constexpr int NI = 64;             // inducers
constexpr int HD = 48;             // head dim
constexpr int NH = 8;              // heads
constexpr int C = NH * HD;         // 384
constexpr int BK = 64;
constexpr int NKB = C / BK;        // 6 k-blocks of K
constexpr int QSLOTS = 4;
constexpr int Q_SLOT_BYTES = TM * BK * 2;  // 16 KiB: 128 rows x 64 columns (48 used)
constexpr int K_KB_BYTES = NI * BK * 2;    //  8 KiB
constexpr int VT_BYTES = C * NI * 2;       // 48 KiB: 384 rows (channels) x 128 B (64 inducers)
constexpr int P_BYTES = TM * NI * 2;       // 16 KiB
constexpr int Y_BYTES = TM * HD * 2;       // 12 KiB: 128 rows x 96 B, dense (the box of the output store)
constexpr int O_COLS = C;
constexpr int TMEM_COLS = 512;
constexpr int THREADS = 128 + 256;
constexpr int SMEM_BYTES = 1024 /*align*/ + QSLOTS * Q_SLOT_BYTES + NKB * K_KB_BYTES + VT_BYTES + 2 * P_BYTES + 2 * Y_BYTES +
                           256 /*barriers*/;
static_assert(SMEM_BYTES <= 232448, "shared memory budget");

struct UParams {
  int tiles_per_cloud, num_tiles, tiles_per_cta;
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
unpool_tc_kernel(const __grid_constant__ CUtensorMap tma_q, const __grid_constant__ CUtensorMap tma_k,
                 const __grid_constant__ CUtensorMap tma_vt, const __grid_constant__ CUtensorMap tma_y, const UParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* sQ = smem;                        // [QSLOTS] Q_h windows
  uint8_t* sK = sQ + QSLOTS * Q_SLOT_BYTES;  // [NKB] K k-blocks
  uint8_t* sVT = sK + NKB * K_KB_BYTES;      // V^T
  uint8_t* sP = sVT + VT_BYTES;              // [2] probabilities of the even / odd head in flight
  uint8_t* sY = sP + 2 * P_BYTES;            // [2] output staging of the even / odd warpgroup
  uint64_t* bars = reinterpret_cast<uint64_t*>(sY + 2 * Y_BYTES);
  uint64_t* q_full = bars;                   // [QSLOTS]
  uint64_t* q_empty = q_full + QSLOTS;       // [QSLOTS] the first product has read the slot
  uint64_t* kv_full = q_empty + QSLOTS;      // K and V^T of the cloud landed
  uint64_t* s_full = kv_full + 1;            // [2] S of an even / odd head is in TMEM
  uint64_t* p_full = s_full + 2;             // [2] P written (and S pulled out of TMEM): 4 warp arrivals
  uint64_t* pv_done = p_full + 2;            // [2] the second product is complete: P is free, O_h is final
  uint64_t* tile_done = pv_done + 2;         // every MMA of a tile is complete (K / V^T may be replaced)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tile_done + 1);

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();
  const int lane = threadIdx.x & 31;
  const int tile_begin = blockIdx.x * p.tiles_per_cta;
  const int tile_end = min(tile_begin + p.tiles_per_cta, p.num_tiles);

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_q);
    tma_prefetch_desc(&tma_k);
    tma_prefetch_desc(&tma_vt);
    tma_prefetch_desc(&tma_y);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < QSLOTS; ++i) {
      mbar_init(&q_full[i], 1);
      mbar_init(&q_empty[i], 1);
    }
    mbar_init(kv_full, 1);
    mbar_init(tile_done, 1);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&s_full[i], 1);
      mbar_init(&p_full[i], 4);
      mbar_init(&pv_done[i], 1);
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

  if (warp == 0 && lane == 0) {
    // ------------------------------------------------------------ TMA producer
    int cloud_loaded = -1;
    uint32_t it = 0, g = 0;  // g: (tile, head) pairs issued
    for (int t = tile_begin; t < tile_end; ++t, ++it) {
      const int cloud = t / p.tiles_per_cloud;
      if (cloud != cloud_loaded) {
        // K / V^T are read by the MMAs of the previous tile: wait for its completion barrier
        if (it > 0) mbar_wait(tile_done, (it - 1) & 1u);
        mbar_arrive_expect_tx(kv_full, NKB * K_KB_BYTES + VT_BYTES);
        for (int kb = 0; kb < NKB; ++kb) tma_load_2d(sK + kb * K_KB_BYTES, &tma_k, kv_full, kb * BK, cloud * NI);
        tma_load_2d(sVT, &tma_vt, kv_full, 0, cloud * C);
        tma_load_2d(sVT + VT_BYTES / 2, &tma_vt, kv_full, 0, cloud * C + C / 2);
        cloud_loaded = cloud;
      }
      for (int h = 0; h < NH; ++h, ++g) {
        const uint32_t slot = g % QSLOTS, use = g / QSLOTS;
        mbar_wait(&q_empty[slot], (use & 1u) ^ 1u);
        mbar_arrive_expect_tx(&q_full[slot], Q_SLOT_BYTES);
        tma_load_2d(sQ + slot * Q_SLOT_BYTES, &tma_q, &q_full[slot], h * HD, t * TM);  // columns past 384 are zero-filled
      }
    }
  } else if (uwarp == 1) {
    // ------------------------------------------------------------ MMA issuer (whole warp, one elected lane issues)
    constexpr uint32_t idesc_s = umma_idesc_bf16(TM, NI);
    constexpr uint32_t idesc_o = umma_idesc_bf16(TM, HD);
    const uint32_t sQ_u = uniform_u32(smem_u32(sQ)), sK_u = uniform_u32(smem_u32(sK));
    const uint32_t sVT_u = uniform_u32(smem_u32(sVT)), sP_u = uniform_u32(smem_u32(sP));
    const uint32_t tmem_u = uniform_u32(tmem_base);
    int cloud_loaded = -1;
    uint32_t it = 0, ncl = 0, gs = 0;  // gs: (tile, head) pairs whose first product has been issued
    auto issue_s = [&](int h) {  // S_h = Q_h K_h^T into S buffer h & 1
      const uint32_t slot = gs % QSLOTS, use = gs / QSLOTS;
      mbar_wait(&q_full[slot], use & 1u);
      tc_fence_after_sync();
      if (elect_one()) {
#pragma unroll
        for (int kk = 0; kk < HD / 16; ++kk) {
          const int col = h * HD + kk * 16;  // column of K
          const uint64_t da = umma_desc_k_sw128(sQ_u + slot * Q_SLOT_BYTES) + 2 * kk;
          const uint64_t db = umma_desc_k_sw128(sK_u + (col / BK) * K_KB_BYTES) + (((col % BK) * 2) >> 4);
          umma_bf16_ss(tmem_u + O_COLS + (h & 1) * NI, da, db, idesc_s, kk ? 1u : 0u);
        }
        umma_commit(&q_empty[slot]);
        umma_commit(&s_full[h & 1]);
      }
      __syncwarp();
      ++gs;
    };
    for (int t = tile_begin; t < tile_end; ++t, ++it) {
      const int cloud = t / p.tiles_per_cloud;
      if (cloud != cloud_loaded) {
        mbar_wait(kv_full, ncl & 1u);
        tc_fence_after_sync();
        cloud_loaded = cloud;
        ++ncl;
      }
      // S buffers: pulled out of TMEM before p_full of their last head (6, 7 of the previous tile) was signalled
      issue_s(0);
      issue_s(1);
      for (int h = 0; h < NH; ++h) {
        const uint32_t w = h & 1u, use = it * (NH / 2) + (h >> 1);  // use index of the warpgroup's S / P buffers
        // O_h of the previous tile was drained before the warpgroup wrote this P (program order of the warpgroup)
        mbar_wait(&p_full[w], use & 1u);
        tc_fence_after_sync();
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < NI / 16; ++kk) {
            const uint64_t da = umma_desc_k_sw128(sP_u + w * P_BYTES) + 2 * kk;
            const uint64_t db = umma_desc_k_sw128(sVT_u + h * (HD * 128)) + 2 * kk;
            umma_bf16_ss(tmem_u + h * HD, da, db, idesc_o, kk ? 1u : 0u);
          }
          umma_commit(&pv_done[w]);
        }
        __syncwarp();
        if (h + 2 < NH) issue_s(h + 2);
      }
      if (elect_one()) umma_commit(tile_done);
      __syncwarp();
    }
  } else if (warp >= 4) {
    // ------------------------------------------------------------ softmax warpgroups + output
    const int w = (warp - 4) >> 2;            // 0: even heads, 1: odd heads
    const int q = warp & 3;                   // TMEM lane quadrant
    const uint32_t row = q * 32 + lane;       // row of the tile owned by this thread
    const uint32_t x7 = (row & 7u) << 4;
    const uint32_t lane_addr = static_cast<uint32_t>(q * 32) << 16;
    const uint32_t p_row = smem_u32(sP) + w * P_BYTES + row * 128u;
    uint8_t* y_stage = sY + w * Y_BYTES;
    const uint32_t y_row = smem_u32(y_stage) + row * (HD * 2);
    const bool storer = (warp & 3) == 0 && lane == 0;  // first thread of the warpgroup issues its bulk stores
    uint32_t use = 0;                         // heads processed by this warpgroup
    float inv_prev = 0.f;
    int t_prev = 0, h_prev = -1;

    // drain O of a finished head: normalise, stage [128 x 48] bf16, one bulk tensor store
    // (the caller has waited for the head's second product: pv_done)
    auto drain = [&](int t_of, int h_of, float inv) {
      uint32_t o[48];
      tmem_ld16(tmem_base + lane_addr + h_of * HD, o);
      tmem_ld16(tmem_base + lane_addr + h_of * HD + 16, o + 16);
      tmem_ld16(tmem_base + lane_addr + h_of * HD + 32, o + 32);
      tmem_ld_wait();
      tc_fence_before_sync();
      if (storer) tma_store_wait_read<0>();     // the previous store of this warpgroup has read the staging buffer
      named_bar_sync(1 + w, 128);
#pragma unroll
      for (int i = 0; i < 6; ++i)
        sts128(y_row + 16u * i,
               pack_bf16x2(__uint_as_float(o[8 * i + 0]) * inv, __uint_as_float(o[8 * i + 1]) * inv),
               pack_bf16x2(__uint_as_float(o[8 * i + 2]) * inv, __uint_as_float(o[8 * i + 3]) * inv),
               pack_bf16x2(__uint_as_float(o[8 * i + 4]) * inv, __uint_as_float(o[8 * i + 5]) * inv),
               pack_bf16x2(__uint_as_float(o[8 * i + 6]) * inv, __uint_as_float(o[8 * i + 7]) * inv));
      fence_proxy_async_smem();
      named_bar_sync(1 + w, 128);
      if (storer) {
        tma_store_2d_addr(&tma_y, smem_u32(y_stage), h_of * HD, t_of * TM);
        tma_store_commit();
      }
    };

    for (int t = tile_begin; t < tile_end; ++t) {
#pragma unroll 1
      for (int j = 0; j < NH / 2; ++j, ++use) {
        const int h = 2 * j + w;
        mbar_wait(&s_full[w], use & 1u);
        tc_fence_after_sync();
        uint32_t s0[32], s1[32];
        tmem_ld32(tmem_base + lane_addr + O_COLS + w * NI, s0);
        tmem_ld32(tmem_base + lane_addr + O_COLS + w * NI + 32, s1);
        tmem_ld_wait();
        float mx = -INFINITY;
#pragma unroll
        for (int i = 0; i < 32; ++i) mx = fmaxf(mx, fmaxf(__uint_as_float(s0[i]), __uint_as_float(s1[i])));
        float sum = 0.f;
        uint32_t pk[32];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a = ex2f(__uint_as_float(s0[2 * i]) - mx), b = ex2f(__uint_as_float(s0[2 * i + 1]) - mx);
          sum += a + b;
          pk[i] = pack_bf16x2(a, b);
        }
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a = ex2f(__uint_as_float(s1[2 * i]) - mx), b = ex2f(__uint_as_float(s1[2 * i + 1]) - mx);
          sum += a + b;
          pk[16 + i] = pack_bf16x2(a, b);
        }
        // the second product of this warpgroup's previous head has read the P buffer
        // (exact: the next completion of this barrier needs the p_full arrival below) -- O of that head is final too
        if (use > 0) {
          mbar_wait(&pv_done[w], (use - 1) & 1u);
          tc_fence_after_sync();
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) sts128(p_row + ((((uint32_t)i) << 4) ^ x7), pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
        fence_proxy_async_smem();
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&p_full[w]);
        // while the tensor core works on this head, write out the previous one
        if (h_prev >= 0) drain(t_prev, h_prev, inv_prev);
        inv_prev = 1.0f / sum;
        t_prev = t;
        h_prev = h;
      }
    }
    if (h_prev >= 0) {
      mbar_wait(&pv_done[w], (use - 1) & 1u);  // the last head: no further completion can follow
      tc_fence_after_sync();
      drain(t_prev, h_prev, inv_prev);
    }
    if (storer) tma_store_wait_read<0>();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

// V^T of every cloud: vt[cloud][c][i] = kv[cloud * 64 + i][v_off + c]  (bf16), through a padded shared-memory tile.
// grid (clouds, 2): one half of the channels per block.
__global__ void __launch_bounds__(256) transpose_v_kernel(const __nv_bfloat16* __restrict__ kv, long long ldkv, int v_off,
                                                          __nv_bfloat16* __restrict__ vt) {
  constexpr int CH = C / 2;
  __shared__ __nv_bfloat16 tile[NI][CH + 8];
  pdl_wait();  // programmatic dependent launch: the predecessor has completed
  pdl_launch_dependents();
  const int cloud = blockIdx.x, c0 = blockIdx.y * CH;
  const __nv_bfloat16* src = kv + (long long)cloud * NI * ldkv + v_off + c0;
  for (int i = threadIdx.x; i < NI * (CH / 8); i += blockDim.x) {
    const int r = i / (CH / 8), c8 = i % (CH / 8);
    *reinterpret_cast<uint4*>(&tile[r][c8 * 8]) = *reinterpret_cast<const uint4*>(src + (long long)r * ldkv + c8 * 8);
  }
  __syncthreads();
  __nv_bfloat16* dst = vt + ((long long)cloud * C + c0) * NI;
  for (int i = threadIdx.x; i < CH * (NI / 2); i += blockDim.x) {
    const int c = i / (NI / 2), i2 = i % (NI / 2);
    __nv_bfloat162 v;
    v.x = tile[2 * i2][c];
    v.y = tile[2 * i2 + 1][c];
    *reinterpret_cast<__nv_bfloat162*>(dst + (long long)c * NI + 2 * i2) = v;
  }
}

}  // namespace

bool unpool_tc_supported(const gecco_unpool_args& a) {
  return a.vt_scratch != nullptr && a.heads == NH && a.head_dim == HD && a.inducers == NI && a.rows_per_cloud % TM == 0 &&
         a.ldq % 8 == 0 && a.ldkv % 8 == 0 && a.ldo % 8 == 0 && a.v_off % 8 == 0 &&
         (reinterpret_cast<uintptr_t>(a.q) & 15) == 0 && (reinterpret_cast<uintptr_t>(a.kv) & 15) == 0 &&
         (reinterpret_cast<uintptr_t>(a.out_bf16) & 15) == 0 && (reinterpret_cast<uintptr_t>(a.vt_scratch) & 15) == 0;
}

int launch_unpool_tc(const gecco_unpool_args& a, cudaStream_t stream) {
  GECCO_REQUIRE(unpool_tc_supported(a), "unpool attention (tcgen05): unsupported shape");
  const long long rows = (long long)a.clouds * a.rows_per_cloud;
  __nv_bfloat16* vt = static_cast<__nv_bfloat16*>(a.vt_scratch);
  if (!a.vt_ready) {
    launch_small(transpose_v_kernel, dim3(a.clouds, 2), dim3(256), 0, stream, static_cast<const __nv_bfloat16*>(a.kv), a.ldkv, a.v_off, vt);
    GECCO_CHECK_LAUNCH("transpose_v_kernel");
  }

  CUtensorMap tq, tk, tvt, ty;
  if (int rc = make_tmap_bf16(&tq, a.q, C, rows, a.ldq, TM)) return rc;
  if (int rc = make_tmap_bf16(&tk, a.kv, C, (uint64_t)a.clouds * NI, a.ldkv, NI)) return rc;
  if (int rc = make_tmap_bf16(&tvt, vt, NI, (uint64_t)a.clouds * C, NI, C / 2)) return rc;
  if (int rc = make_tmap(&ty, 2, a.out_bf16, C, rows, (uint64_t)a.ldo * 2, HD, TM, 0)) return rc;  // dense [128 x 48] boxes

  UParams p;
  p.tiles_per_cloud = a.rows_per_cloud / TM;
  p.num_tiles = a.clouds * p.tiles_per_cloud;
  const int sms = sm_count();
  p.tiles_per_cta = ceil_div(p.num_tiles, sms);
  const int grid = ceil_div(p.num_tiles, p.tiles_per_cta);

  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(unpool_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(unpool_tc_kernel)");
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
  cudaError_t le = cudaLaunchKernelEx(&cfg, unpool_tc_kernel, tq, tk, tvt, ty, p);
  if (le != cudaSuccess) return fail_cuda(le, "unpool_tc_kernel launch");
  GECCO_CHECK_LAUNCH("unpool_tc_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco
