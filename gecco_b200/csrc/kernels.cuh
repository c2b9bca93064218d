// Internal launcher declarations shared between the per-kernel translation units and engine.cu.
#pragma once
#include "common.cuh"

#include <cuda.h>

namespace gecco {

// tensor-map builders (gemm_tc.cu)
int make_tmap(CUtensorMap* m, int elem_bytes, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld_bytes,
              uint32_t box_cols, uint32_t box_rows, int swizzle);
int make_tmap_bf16(CUtensorMap* m, const void* ptr, uint64_t cols, uint64_t rows, uint64_t ld, uint32_t box_rows);
int make_output_tmaps(float* o32, long long ldo32, void* o16, long long ldo16, int m, int n_out, const CUtensorMap& dummy,
                      CUtensorMap* t32, CUtensorMap* t16);
int make_residual_tmap(const float* res, long long ldr, int m, int n_out, const CUtensorMap& dummy, CUtensorMap* tres);
// CTA-pair (cta_group::2) variant of the GEMM for K <= 384 with the A tile resident in shared memory (gemm_pair.cu).
// Returns GECCO_OK and sets *handled = 1 when the problem fits, *handled = 0 when the caller must use launch_gemm's
// single-CTA kernel.
int launch_gemm_pair(const gecco_gemm_args& a, cudaStream_t s, int* handled);
// A-operand AdaGN (gecco_anorm) is available for this shape (CTA-pair kernel, k % 64 == 0) and the pair kernel is enabled.
bool gemm_anorm_supported(int m, int rows_per_cloud, int n_out, int k);
bool g_use_pairs_ref();
void set_fast_epilogue_option(int value);  // gemm_pair.cu: gecco_set_option("fast_epilogue", v)

int launch_gemm(const gecco_gemm_args& a, cudaStream_t s);
void set_graphs_option(int value);  // engine.cu: gecco_set_option("graphs", v)
void set_chain_option(int value);  // engine.cu: gecco_set_option("chain", v)
void set_anorm_option(int value);  // engine.cu: gecco_set_option("anorm", v)
// CTA-pair MLP with the hidden tile parked in an L2-resident scratch and AdaGN on the A operand (mlp_pair.cu).
bool mlp_pair_supported(const gecco_mlp_args& a);
int launch_mlp_pair(const gecco_mlp_args& a, cudaStream_t s);
void set_mlp_pair_option(int value);  // engine.cu: gecco_set_option("mlp_pair", v)
int launch_group_stats(const float* x, long long ldx, int clouds, int rows_per_cloud, int valid_rows, int C, int gs,
                       double* stats, cudaStream_t s);
int launch_adagn(const gecco_adagn_args& a, cudaStream_t s);
int launch_fold_adagn(const gecco_fold_adagn_args& a, cudaStream_t s);
int launch_lift(const gecco_lift_args& a, cudaStream_t s);
int launch_head(const gecco_head_args& a, cudaStream_t s);
int launch_sampler_init(const float* latents, const float* noise, double t0, double churn, long long n, double* x_hat,
                        float* xin, cudaStream_t s);
int launch_seed_renoise(const float* data, const float* noise, float t, long long n, float* out, cudaStream_t s);
int launch_substep_noise(const double* src, const float* n1, float c1, const float* n2, float c2, long long n, double* x_hat,
                         float* xin, cudaStream_t s);
int launch_lookup(const gecco_lookup_args& a, cudaStream_t s);
int launch_fold_gn(const float* W, const float* bias, const double* stats, double count, float eps, int groups,
                   int c_in, int c_out, int clouds, void* wb, long long ldwb, float* bb, cudaStream_t s);
int launch_pool_attention(const gecco_pool_args& a, cudaStream_t s);
int launch_unpool_attention(const gecco_unpool_args& a, cudaStream_t s);
// tcgen05 / TMEM version of the unpool attention core (attention_tc.cu); needs a.vt_scratch.
bool unpool_tc_supported(const gecco_unpool_args& a);
int launch_unpool_tc(const gecco_unpool_args& a, cudaStream_t s);

// tcgen05 / TMEM version of the pool attention core (attention_pool_tc.cu).  *splits_used > 1: the result was left as
// key-split partials in a.partial (pool_combine_kernel finishes); 1: a.out_bf16 is final.
bool pool_tc_supported(const gecco_pool_args& a);
int launch_pool_tc(const gecco_pool_args& a, cudaStream_t s, int* splits_used);

// Inducer side of a Broadcast layer in one cluster kernel (inducer_chain.cu).
bool inducer_chain_supported(const gecco_chain_args& a);
int launch_inducer_chain(const gecco_chain_args& a, cudaStream_t s);
// Pool attention without the final merge of the key splits: *splits_used > 1 means a.partial holds the partials (the
// inducer chain merges them), 1 means a.out_bf16 is final.
int launch_pool_attention_partial(const gecco_pool_args& a, cudaStream_t s, int* splits_used);

}  // namespace gecco
