// Persistent, warp-specialised tcgen05 GEMM with a fused, TMA-staged epilogue (gecco_gemm).
//
//   warp 0 : TMA producer  (A tile 128x64 + W tile 192x64 bf16 per stage, SWIZZLE_128B)
//   warp 1 : MMA issuer    (one thread; 4 x tcgen05.mma M=128 N=192 K=16 per stage)
//   warp 2 : TMEM allocator (512 columns = two 192-wide fp32 accumulator slots)
//   warp 3 : residual loader (TMA prefetch of the fp32 residual chunks the epilogue will add)
//   warps 4-11 : epilogue  (epilogue.cuh: tcgen05.ld -> bias / xyz-embed / activation / residual /
//                           AdaGN statistics -> swizzled smem staging -> TMA bulk stores, fp32 and/or bf16;
//                           two groups of 4 warps on alternate 32-column chunks)
// The two TMEM slots let the epilogue of tile i overlap the main loop of tile i+1.
#include "common.cuh"
#include "epilogue.cuh"
#include "kernels.cuh"
#include "ptx.cuh"

#include <cudaTypedefs.h>
#include <math.h>
#include <string.h>
#include <unordered_map>

namespace gecco {

namespace {

constexpr int BM = 128;
constexpr int BN = 192;
constexpr int BK = 64;
constexpr int MAX_STAGES = 5;  // ring depth is chosen per launch from the shared memory the epilogue leaves
constexpr int A_STAGE_BYTES = BM * BK * 2;  // 16 KiB
constexpr int B_STAGE_BYTES = BN * BK * 2;  // 24 KiB
constexpr int ACC_COLS = 256;               // TMEM columns reserved per accumulator slot
constexpr int TMEM_COLS = 512;
constexpr int GEMM_THREADS = 128 + EPI_GROUPS * EPI_THREADS;
constexpr int SMEM_LIMIT = 232448;
constexpr int SMEM_FIXED = 1024 /*align*/ + 256 /*barriers*/;

struct KParams {
  EpiParams e;
  int K, w_rows_per_cloud;
  int num_m_blocks, num_n_blocks;
  int stages;
};

template <bool kStats>
__global__ void __launch_bounds__(GEMM_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w,
               const __grid_constant__ CUtensorMap tma_res, const __grid_constant__ CUtensorMap tma_o32,
               const __grid_constant__ CUtensorMap tma_o16, const KParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int STAGES = p.stages;
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * A_STAGE_BYTES;
  uint8_t* sEpi = smem + STAGES * (A_STAGE_BYTES + B_STAGE_BYTES);
  EpiSmem es;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_smem_carve(es, sEpi, p.e.has_res, p.e.o32 != nullptr, p.e.o16 != nullptr));
  uint64_t* full_bar = bars;                 // [MAX_STAGES]
  uint64_t* empty_bar = bars + MAX_STAGES;   // [MAX_STAGES]
  uint64_t* acc_full = bars + 2 * MAX_STAGES;    // [2]
  uint64_t* acc_empty = bars + 2 * MAX_STAGES + 2;  // [2]  one arrival per epilogue warp
  es.res_full = bars + 2 * MAX_STAGES + 4;   // [EPI_GROUPS][2]
  es.res_empty = es.res_full + EPI_NUM_BARS / 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(es.res_full + EPI_NUM_BARS);

  const int warp = threadIdx.x >> 5;
  const int uwarp = uniform_warp_idx();  // same value, provably warp-uniform (all threads converged here)
  const int lane = threadIdx.x & 31;
  const int num_tiles = p.num_m_blocks * p.num_n_blocks;
  const int num_kb = (p.K + BK - 1) / BK;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    if (p.e.has_res) tma_prefetch_desc(&tma_res);
    if (p.e.o32 != nullptr) tma_prefetch_desc(&tma_o32);
    if (p.e.o16 != nullptr) tma_prefetch_desc(&tma_o16);
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < MAX_STAGES; ++i) {
      mbar_init(&full_bar[i], 1);
      mbar_init(&empty_bar[i], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], EPI_GROUPS * EPI_THREADS / 32);
    }
    epi_bar_init(es);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<TMEM_COLS>(tmem_slot);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = *tmem_slot;
  // everything above overlaps the tail of the preceding kernel (programmatic dependent launch)
  pdl_wait();
  pdl_launch_dependents();

  // warps 0-3 (TMA / MMA / allocator / residual loader: a handful of registers) hand their registers to the epilogue
  if (warp < 4) {
  setmaxnreg_dec<40>();
  if (warp == 0 && lane == 0) {
    // ------------------------------------------------------------ TMA producer
    int stage = 0;
    uint32_t phase = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
      const int m0 = (t / p.num_n_blocks) * BM;
      const int n0 = (t % p.num_n_blocks) * BN;
      const int wrow = (p.w_rows_per_cloud ? (m0 / p.e.rows_per_cloud) * p.w_rows_per_cloud : 0) + n0;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        mbar_arrive_expect_tx(&full_bar[stage], A_STAGE_BYTES + B_STAGE_BYTES);
        tma_load_2d(sA + stage * A_STAGE_BYTES, &tma_a, &full_bar[stage], kb * BK, m0);
        tma_load_2d(sB + stage * B_STAGE_BYTES, &tma_w, &full_bar[stage], kb * BK, wrow);
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
    }
  } else if (uwarp == 1) {
    // ------------------------------------------------------------ MMA issuer: the whole warp runs the loop (uniform
    // control flow keeps the descriptors in uniform registers, see ptx.cuh), one elected lane issues
    constexpr uint32_t idesc = umma_idesc_bf16(BM, BN);
    const uint32_t sA_u = uniform_u32(smem_u32(sA)), sB_u = uniform_u32(smem_u32(sB));
    const uint32_t tmem_u = uniform_u32(tmem_base);
    int stage = 0;
    uint32_t phase = 0;
    int it = 0;
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int slot = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&acc_empty[slot], acc_phase ^ 1);
      tc_fence_after_sync();
      const uint32_t tmem_d = tmem_u + slot * ACC_COLS;
      for (int kb = 0; kb < num_kb; ++kb) {
        mbar_wait(&full_bar[stage], phase);
        tc_fence_after_sync();
        const uint64_t da = umma_desc_k_sw128(sA_u + stage * A_STAGE_BYTES);
        const uint64_t db = umma_desc_k_sw128(sB_u + stage * B_STAGE_BYTES);
        if (elect_one()) {
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            // +32 B per K=16 step inside the 128 B swizzle row (address field is in 16 B units)
            umma_bf16_ss(tmem_d, da + 2 * k, db + 2 * k, idesc, (kb | k) ? 1u : 0u);
          }
          umma_commit(&empty_bar[stage]);
        }
        __syncwarp();
        if (++stage == STAGES) { stage = 0; phase ^= 1; }
      }
      if (elect_one()) umma_commit(&acc_full[slot]);
      __syncwarp();
    }
  } else if (warp == 3 && lane == 0) {
    // ------------------------------------------------------------ residual loader
    if (p.e.has_res) {
      uint32_t cnt[EPI_GROUPS] = {0, 0};
      for (int t = blockIdx.x; t < num_tiles; t += gridDim.x) {
        const int m0 = (t / p.num_n_blocks) * BM;
        const int n0 = (t % p.num_n_blocks) * BN;
        epi_load_residual_panel(p.e, es, &tma_res, m0, n0, cnt);
      }
    }
  }
  } else {
    setmaxnreg_inc<232>();
    // ------------------------------------------------------------ epilogue
    const EpiThread et = epi_thread_init(es, (warp - 4) >> 2, threadIdx.x & (EPI_THREADS - 1));
    const int q = warp & 3;  // TMEM lane quadrant of this warp
    int it = 0;
    uint32_t cnt = 0;
    EpiBias bias_r;
    if ((int)blockIdx.x < num_tiles)
      epi_bias_load(p.e, et, ((int)blockIdx.x / p.num_n_blocks) * BM, ((int)blockIdx.x % p.num_n_blocks) * BN, bias_r);
    for (int t = blockIdx.x; t < num_tiles; t += gridDim.x, ++it) {
      const int slot = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int m0 = (t / p.num_n_blocks) * BM;
      const int n0 = (t % p.num_n_blocks) * BN;
      epi_bias_stage(p.e, et, bias_r);
      const int tn = t + gridDim.x;  // the next tile's bias is loaded under this tile
      if (tn < num_tiles) epi_bias_load(p.e, et, (tn / p.num_n_blocks) * BM, (tn % p.num_n_blocks) * BN, bias_r);
      mbar_wait(&acc_full[slot], acc_phase);
      tc_fence_after_sync();
      const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16) + slot * ACC_COLS;
      epi_panel<kStats>(p.e, es, et, &tma_o32, &tma_o16, taddr, m0, n0, cnt);
      tc_fence_before_sync();
      __syncwarp();
      if (et.lane == 0) mbar_arrive(&acc_empty[slot]);  // one arrival per warp
    }
    if (et.lane == 0) tma_store_wait_read<0>();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after_sync();
    tmem_dealloc<TMEM_COLS>(tmem_base);
  }
}

PFN_cuTensorMapEncodeTiled g_encode = nullptr;
bool g_use_pairs = true;
int g_epi_skip = 0;  // gecco_set_option("gemm_pairs", 0) selects the single-CTA kernel everywhere

}  // namespace
int epi_skip_option() { return g_epi_skip; }

int resolve_driver() {
  if (g_encode != nullptr) return GECCO_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || fn == nullptr || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled not available from the driver");
    return GECCO_ERR_CUDA;
  }
  g_encode = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(fn);
  return GECCO_OK;
}

int make_tmap_uncached(CUtensorMap* m, int elem_bytes, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_bytes,
                       uint32_t box_cols, uint32_t box_rows, int swizzle);

// Row-major [rows, cols] matrix (ld_bytes between rows) viewed as a 2D tensor {cols, rows} with a
// {box_cols, box_rows} box.  swizzle: 128 / 64 (bytes) - the box row must span exactly that many bytes or less.
// cuTensorMapEncodeTiled costs several microseconds and the engine asks for the same few dozen maps on every
// evaluation (the workspace is stable), so encoded maps are cached per thread.
struct TmapKey {
  const void* ptr;
  uint64_t cols, rows, ld_bytes;
  uint32_t box_cols, box_rows;
  int elem_bytes, swizzle;
  bool operator==(const TmapKey& o) const {
    return ptr == o.ptr && cols == o.cols && rows == o.rows && ld_bytes == o.ld_bytes && box_cols == o.box_cols &&
           box_rows == o.box_rows && elem_bytes == o.elem_bytes && swizzle == o.swizzle;
  }
};
struct TmapKeyHash {
  size_t operator()(const TmapKey& k) const {
    uint64_t h = reinterpret_cast<uintptr_t>(k.ptr) * 0x9E3779B97F4A7C15ull;
    h ^= (k.cols + 0x9E3779B97F4A7C15ull + (h << 6) + (h >> 2));
    h ^= (k.rows * 0xC2B2AE3D27D4EB4Full + (h << 6) + (h >> 2));
    h ^= (k.ld_bytes * 0x165667B19E3779F9ull + (h << 6) + (h >> 2));
    h ^= ((uint64_t)k.box_cols << 40) ^ ((uint64_t)k.box_rows << 24) ^ ((uint64_t)k.elem_bytes << 8) ^ (uint64_t)k.swizzle;
    return static_cast<size_t>(h);
  }
};
static thread_local std::unordered_map<TmapKey, CUtensorMap, TmapKeyHash> t_tmap_cache;

int make_tmap(CUtensorMap* m, int elem_bytes, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_bytes,
              uint32_t box_cols, uint32_t box_rows, int swizzle) {
  const TmapKey key{ptr, cols, rows, ld_bytes, box_cols, box_rows, elem_bytes, swizzle};
  auto hit = t_tmap_cache.find(key);
  if (hit != t_tmap_cache.end()) {
    *m = hit->second;
    return GECCO_OK;
  }
  if (int rc = make_tmap_uncached(m, elem_bytes, ptr, cols, rows, ld_bytes, box_cols, box_rows, swizzle)) return rc;
  if (t_tmap_cache.size() > 8192) t_tmap_cache.clear();
  t_tmap_cache.emplace(key, *m);
  return GECCO_OK;
}

int make_tmap_uncached(CUtensorMap* m, int elem_bytes, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_bytes,
                       uint32_t box_cols, uint32_t box_rows, int swizzle) {
  if (int rc = resolve_driver()) return rc;
  GECCO_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "operand pointer must be 16-byte aligned");
  GECCO_REQUIRE(ld_bytes % 16 == 0, "operand leading dimension must be a multiple of 16 bytes (got %llu)",
                (unsigned long long)ld_bytes);
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {ld_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapDataType dt = elem_bytes == 2 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
  const CUtensorMapSwizzle sw = swizzle == 128 ? CU_TENSOR_MAP_SWIZZLE_128B
                                : swizzle == 64 ? CU_TENSOR_MAP_SWIZZLE_64B
                                : swizzle == 32 ? CU_TENSOR_MAP_SWIZZLE_32B : CU_TENSOR_MAP_SWIZZLE_NONE;
  CUresult r = g_encode(m, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, sw,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (cols=%llu rows=%llu ld=%llu B box=%ux%u)", (int)r,
              (unsigned long long)cols, (unsigned long long)rows, (unsigned long long)ld_bytes, box_cols, box_rows);
    return GECCO_ERR_CUDA;
  }
  return GECCO_OK;
}

// bf16 MMA operand: box {64, box_rows}, SWIZZLE_128B.
int make_tmap_bf16(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_rows) {
  GECCO_REQUIRE(ld % 8 == 0, "operand leading dimension must be a multiple of 8 elements (got %llu)", (unsigned long long)ld);
  return make_tmap(m, 2, ptr, cols, rows, ld * 2, 64, box_rows, 128);
}

// Tensor map of the epilogue's residual prefetch (epilogue.cuh): fp32 chunks {32, 128}, SWIZZLE_128B.  Without a
// residual the map is a copy of `dummy` (never dereferenced).
int make_residual_tmap(const float* res, long long ldr, int m, int n_out, const CUtensorMap& dummy, CUtensorMap* tres) {
  *tres = dummy;
  GECCO_REQUIRE(!res || ldr % 4 == 0, "residual leading dimension must be a multiple of 4");
  if (res) return make_tmap(tres, 4, res, n_out, m, ldr * 4, EPI_CHUNK, 128, 128);
  return GECCO_OK;
}

// Tensor maps of the epilogue's per-warp bulk stores: {32 columns, 32 rows} boxes, SWIZZLE_128B (fp32) / SWIZZLE_64B (bf16).
int make_output_tmaps(float* o32, long long ldo32, void* o16, long long ldo16, int m, int n_out, const CUtensorMap& dummy,
                      CUtensorMap* t32, CUtensorMap* t16) {
  *t32 = dummy; *t16 = dummy;
  GECCO_REQUIRE(!o32 || ldo32 % 4 == 0, "fp32 output leading dimension must be a multiple of 4");
  GECCO_REQUIRE(!o16 || ldo16 % 8 == 0, "bf16 output leading dimension must be a multiple of 8");
  if (o32) if (int rc = make_tmap(t32, 4, o32, n_out, m, ldo32 * 4, EPI_CHUNK, 32, 128)) return rc;
  if (o16) if (int rc = make_tmap(t16, 2, o16, n_out, m, ldo16 * 2, EPI_CHUNK, 32, 64)) return rc;
  return GECCO_OK;
}

int launch_gemm(const gecco_gemm_args& a, cudaStream_t stream) {
  GECCO_REQUIRE(a.w, "gemm: null operand");
  GECCO_REQUIRE(a.m > 0 && a.n_out > 0 && a.k > 0, "gemm: empty problem m=%d n=%d k=%d", a.m, a.n_out, a.k);
  GECCO_REQUIRE(a.n_out % 8 == 0, "gemm: n_out (%d) must be a multiple of 8", a.n_out);
  GECCO_REQUIRE(a.rows_per_cloud > 0 && a.rows_per_cloud % 32 == 0, "gemm: rows_per_cloud (%d) must be a positive multiple of 32",
                a.rows_per_cloud);
  GECCO_REQUIRE(a.valid_rows > 0 && a.valid_rows <= a.rows_per_cloud, "gemm: valid_rows out of range");
  GECCO_REQUIRE(a.out_f32 || a.out_bf16, "gemm: no output buffer");
  GECCO_REQUIRE(!a.stats || a.n_out % 12 == 0, "gemm: statistics epilogue needs n_out %% 12 == 0");
  GECCO_REQUIRE(!a.geom || (a.sigma && a.wx), "gemm: xyz embed needs sigma and wx");
  GECCO_REQUIRE(!a.w_rows_per_cloud || a.rows_per_cloud % BM == 0,
                "gemm: per-cloud weights need rows_per_cloud %% 128 == 0");

  GECCO_REQUIRE(a.anorm.stats == nullptr || gemm_anorm_supported(a.m, a.rows_per_cloud, a.n_out, a.k),
                "gemm: A-operand normalisation is not available for this shape (m=%d rows_per_cloud=%d n_out=%d k=%d): see "
                "gecco_gemm_anorm_supported", a.m, a.rows_per_cloud, a.n_out, a.k);
  GECCO_REQUIRE(a.a != nullptr, "gemm: null operand");
  if (g_use_pairs) {
    int handled = 0;
    if (int rc = launch_gemm_pair(a, stream, &handled)) return rc;
    if (handled) return GECCO_OK;
  }
  const int clouds = ceil_div(a.m, a.rows_per_cloud);
  const uint64_t w_rows = a.w_rows_per_cloud ? (uint64_t)a.w_rows_per_cloud * (clouds - 1) + a.n_out : (uint64_t)a.n_out;
  CUtensorMap ta, tw, tres, t32, t16;
  if (int rc = make_tmap_bf16(&ta, a.a, a.k, a.m, a.lda, BM)) return rc;
  if (int rc = make_tmap_bf16(&tw, a.w, a.k, w_rows, a.ldw, BN)) return rc;
  if (int rc = make_residual_tmap(a.res, a.ldr, a.m, a.n_out, ta, &tres)) return rc;
  if (int rc = make_output_tmaps(a.out_f32, a.ldo32, a.out_bf16, a.ldo16, a.m, a.n_out, ta, &t32, &t16)) return rc;

  KParams p;
  p.e.M = a.m; p.e.n_out = a.n_out; p.K = a.k;
  p.e.rows_per_cloud = a.rows_per_cloud; p.e.valid_rows = a.valid_rows; p.w_rows_per_cloud = a.w_rows_per_cloud;
  p.e.bias = a.bias; p.e.bias_stride = a.bias_stride;
  p.e.act = a.act;
  p.e.act_k = a.act ? static_cast<float>(-1.4426950408889634 / (2.0 * (double)a.act_alpha * (double)a.act_alpha)) : 0.f;
  p.e.has_res = a.res != nullptr;
  p.e.o32 = a.out_f32;
  p.e.o16 = static_cast<__nv_bfloat16*>(a.out_bf16);
  p.e.stats = a.stats;
  p.e.geom = a.geom; p.e.sigma = a.sigma; p.e.sigma_stride = a.sigma_stride; p.e.sigma_data = a.sigma_data; p.e.wx = a.wx;
  p.e.dbg = nullptr;
  p.e.skip = 0;
  p.e.hints = 0;
  p.num_m_blocks = ceil_div(a.m, BM);
  p.num_n_blocks = ceil_div(a.n_out, BN);
  const int epi_bytes = epi_smem_bytes(p.e.has_res, a.out_f32 != nullptr, a.out_bf16 != nullptr);
  p.stages = (SMEM_LIMIT - SMEM_FIXED - epi_bytes) / (A_STAGE_BYTES + B_STAGE_BYTES);
  if (p.stages > MAX_STAGES) p.stages = MAX_STAGES;
  const int smem_bytes = SMEM_FIXED + epi_bytes + p.stages * (A_STAGE_BYTES + B_STAGE_BYTES);

  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(gemm_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(gemm_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT);
    if (e != cudaSuccess) return fail_cuda(e, "cudaFuncSetAttribute(gemm_tc_kernel)");
    attr_set = true;
  }
  const int tiles = p.num_m_blocks * p.num_n_blocks;
  const int grid = tiles < sm_count() ? tiles : sm_count();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  cudaError_t le = a.stats ? cudaLaunchKernelEx(&cfg, gemm_tc_kernel<true>, ta, tw, tres, t32, t16, p)
                           : cudaLaunchKernelEx(&cfg, gemm_tc_kernel<false>, ta, tw, tres, t32, t16, p);
  if (le != cudaSuccess) return fail_cuda(le, "gemm_tc_kernel launch");
  GECCO_CHECK_LAUNCH("gemm_tc_kernel launch");
  return GECCO_OK;
}

}  // namespace gecco

namespace gecco {
bool g_use_pairs_ref() { return g_use_pairs; }
}  // namespace gecco

extern "C" int gecco_gemm_anorm_supported(int32_t m, int32_t rows_per_cloud, int32_t n_out, int32_t k) {
  return gecco::gemm_anorm_supported(m, rows_per_cloud, n_out, k) ? 1 : 0;
}

extern "C" int gecco_set_option(const char* name, int value) {
  if (name != nullptr && strcmp(name, "gemm_pairs") == 0) {
    gecco::g_use_pairs = value != 0;
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "epi_skip") == 0) {
    gecco::g_epi_skip = value;
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "fast_epilogue") == 0) {
    gecco::set_fast_epilogue_option(value);
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "anorm") == 0) {
    gecco::set_anorm_option(value);
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "mlp_pair") == 0) {
    gecco::set_mlp_pair_option(value);
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "chain") == 0) {
    gecco::set_chain_option(value);
    return GECCO_OK;
  }
  if (name != nullptr && strcmp(name, "graphs") == 0) {
    gecco::set_graphs_option(value);
    return GECCO_OK;
  }
  gecco::set_error("gecco_set_option: unknown option '%s'", name ? name : "(null)");
  return GECCO_ERR_INVALID;
}

extern "C" int gecco_gemm(const gecco_gemm_args* args, void* stream) {
  if (args == nullptr) {
    gecco::set_error("gecco_gemm: null args");
    return GECCO_ERR_INVALID;
  }
  return gecco::launch_gemm(*args, static_cast<cudaStream_t>(stream));
}
