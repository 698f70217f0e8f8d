// Host-side interface of the tcgen05 GEMM (used by the engine and by the C-ABI).
#pragma once
#include "gemm_tcgen05.cuh"

namespace vq {

struct GemmOperand {
  const void* ptr;  // bf16
  int ld;           // pitch in elements of the stored 2-D tensor
  bool mn_major;    // false: stored [MN rows, K contiguous]; true: stored [K rows, MN contiguous]
};

// C[M,N] (+)= A[M,K] * B[N,K]^T with the epilogue in args.epi. force_bn = 0 picks the N tile by occupancy.
int gemm_bf16(const GemmOperand& A, const GemmOperand& B, GemmArgs args, int force_bn, cudaStream_t stream);
// split-K factor gemm_bf16 really uses for a request of `splits` over K: clamped to the 64-deep k-blocks and rounded so that
// no split is empty (a consumer of the split_stride slabs must add exactly this many)
int gemm_split_count(int K, int splits);
// n <= GEMM_GROUP_MAX independent weight-gradient problems C_i[M_i, N_i] += A_i[M_i, K] * B_i[N_i, K]^T (both operands MN-major,
// shared K) as ONE launch of the CTA-pair kernel; epi = EPI_ATOMIC_F32 (accumulate) or EPI_F32 (store)
struct GemmGroupProblem {
  const void* A; int lda;     // stored [K, M]
  const void* B; int ldb;     // stored [K, N]
  void* C; int ldc;           // fp32 [M, N]
  int M, N;
};
int gemm_bf16_grouped_mn(const GemmGroupProblem* probs, int n, int K, int epi, float alpha, int sm_limit, cudaStream_t stream);
bool gemm_pair_on();            // CTA-pair kernel available (VQACL_GEMM_PAIR=0 turns it off for A/B runs): needed by the grouped form
bool gemm_vis_tail_on();        // VisualEmbedding as ONE launch (GEMM + row tail 2); VQACL_VIS_FUSED=0 keeps GEMM + vis_embed_fwd_kernel
bool gemm_row_tail_ok(int M);   // fold a row-wise follow-up (RMSNorm) into a GEMM with 768 output columns? (see gemm.cu)
void gemm_tmap_cache_clear();
// cached 2-D bf16 tensor map, 128-byte swizzle: inner extent d0 (contiguous), outer extent d1, outer pitch ld elements, box b0 x b1
int make_tmap_bf16_2d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t ld, uint32_t b0, uint32_t b1);
int num_sms();

}  // namespace vq
