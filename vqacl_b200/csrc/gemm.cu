// Host side of the tcgen05 GEMM: TMA tensor-map construction (cuTensorMapEncodeTiled through the
// runtime's driver entry point, so the library does not link libcuda), tile-shape selection and launch.
#include "gemm.h"

#include <cudaTypedefs.h>
#include <mutex>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>
#include <unordered_map>

// ------------------------------------------------------------------------------------------
// error channel shared by the whole library
// ------------------------------------------------------------------------------------------
static thread_local char g_err[1024] = "";
void vq_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
extern "C" const char* vqacl_last_error() { return g_err; }
long long g_vq_launches = 0;
// VQACL_NO_PDL=1: plain stream ordering for every launch (measurement only: with PDL a kernel's CUPTI duration includes
// the time it waits for its predecessor, so per-kernel timelines are taken with this set)
int g_vq_pdl = [] { const char* e = getenv("VQACL_NO_PDL"); return (e && e[0] == '1') ? 0 : 1; }();
void vq_kernel_first_use(const void* kern) {
  static std::mutex mu;
  static std::unordered_map<const void*, bool> seen;
  std::lock_guard<std::mutex> g(mu);
  if (seen.emplace(kern, true).second) cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
}
extern "C" long long vqacl_launch_count() { return g_vq_launches; }

namespace vq {

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  });
  return fn;
}

struct TmKey {
  const void* ptr;
  uint64_t d0, d1, ld;
  uint32_t b0, b1;
  bool operator==(const TmKey& o) const {
    return ptr == o.ptr && d0 == o.d0 && d1 == o.d1 && ld == o.ld && b0 == o.b0 && b1 == o.b1;
  }
};
struct TmHash {
  size_t operator()(const TmKey& k) const {
    size_t h = reinterpret_cast<size_t>(k.ptr);
    h = h * 1000003u ^ k.d0;
    h = h * 1000003u ^ k.d1;
    h = h * 1000003u ^ k.ld;
    h = h * 1000003u ^ (((uint64_t)k.b0 << 32) | k.b1);
    return h;
  }
};
static std::unordered_map<TmKey, CUtensorMap, TmHash> g_tm_cache;
static std::mutex g_tm_mutex;

// 2-D bf16 tensor, inner (contiguous) extent d0, outer extent d1, outer pitch ld elements; box b0 x b1, 128 B swizzle.
static int make_tmap(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t ld, uint32_t b0, uint32_t b1) {
  TmKey key{ptr, d0, d1, ld, b0, b1};
  {
    std::lock_guard<std::mutex> g(g_tm_mutex);
    auto it = g_tm_cache.find(key);
    if (it != g_tm_cache.end()) {
      *out = it->second;
      return 0;
    }
  }
  auto fn = get_encode_fn();
  VQ_CHECK(fn != nullptr, "cuTensorMapEncodeTiled entry point not available (driver too old / no GPU)");
  VQ_CHECK((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand base %p is not 16-byte aligned", ptr);
  VQ_CHECK((ld * 2) % 16 == 0, "TMA operand pitch %llu elements is not a multiple of 16 bytes", (unsigned long long)ld);
  cuuint64_t dims[2] = {d0, d1};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {b0, b1};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  VQ_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (dims %llu x %llu, ld %llu, box %u x %u)",
           (int)r, (unsigned long long)d0, (unsigned long long)d1, (unsigned long long)ld, b0, b1);
  {
    std::lock_guard<std::mutex> g(g_tm_mutex);
    if (g_tm_cache.size() > 65536) g_tm_cache.clear();
    g_tm_cache.emplace(key, *out);
  }
  return 0;
}

// shared with the tcgen05 attention kernels (attention_tc.cu)
int make_tmap_bf16_2d(CUtensorMap* out, const void* ptr, uint64_t d0, uint64_t d1, uint64_t ld, uint32_t b0, uint32_t b1) {
  return make_tmap(out, ptr, d0, d1, ld, b0, b1);
}

void gemm_tmap_cache_clear() {
  std::lock_guard<std::mutex> g(g_tm_mutex);
  g_tm_cache.clear();
}

static int g_pair_enabled = 1;   // VQACL_GEMM_PAIR=0 disables the CTA-pair kernel (A/B measurements)
// the engine folds the encoder's sub-layer-opening RMSNorms into the preceding residual GEMMs only on request
// (VQACL_GEMM_ROW_TAIL=1): measured neutral at B = 320 (profiles/r02_summary.md) — 8 tail warps per SM pay the L2 latency of
// 16 rows each, about what the stand-alone kernel costs
static int g_row_tail_off = [] { const char* e = getenv("VQACL_GEMM_ROW_TAIL"); return (e && e[0] == '1') ? 0 : 1; }();
// SMs the persistent GEMMs may occupy (0 = all). With N > 1 GPUs the host lowers it during backward so that the NCCL
// all-reduce kernels, which need resident CTAs of their own, are not starved by 148 GEMM CTAs that each fill an SM's
// shared memory (vqacl_set_gemm_sm_limit).
static int g_sm_limit = 0;
static int g_num_sms = 0;
static int gemm_sms(int call_limit = 0);
int num_sms() {
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
    if (g_num_sms <= 0) g_num_sms = 148;
    const char* ev = getenv("VQACL_GEMM_PAIR");
    if (ev && ev[0] == '0') g_pair_enabled = 0;
  }
  return g_num_sms;
}

static int gemm_sms(int call_limit) {
  int n = num_sms();
  if (g_sm_limit > 0 && g_sm_limit < n) n = g_sm_limit;
  if (call_limit > 0 && call_limit < n) n = call_limit & ~1;   // even: the CTA-pair kernel launches clusters of two
  return n;
}
// Is folding a row tail into an M-row GEMM with 768 output columns a good deal? In the tail mode a CTA pair owns whole 256-row
// blocks, so the kernel's parallelism is ceil(M / 256) pairs instead of 3x as many tiles: only when the blocks fill the pairs
// about as well as the tiles would (B = 320: 70 blocks on 74 pairs either way).
bool gemm_pair_on() {
  (void)num_sms();
  return g_pair_enabled != 0;
}
bool gemm_vis_tail_on() {
  static const int on = [] { const char* e = getenv("VQACL_VIS_FUSED"); return (e && e[0] == '0') ? 0 : 1; }();
  (void)num_sms();
  return on && g_pair_enabled;
}
bool gemm_row_tail_ok(int M) {
  (void)num_sms();
  if (!g_pair_enabled || g_row_tail_off) return false;
  const int pairs = gemm_sms() / 2;
  const int blocks = (M + 255) / 256, tiles = blocks * 3;
  const double eff_own = (double)blocks / ((double)((blocks + pairs - 1) / pairs) * pairs);
  const double eff_tiles = (double)tiles / ((double)((tiles + pairs - 1) / pairs) * pairs);
  return eff_own >= eff_tiles - 0.02;
}

extern "C" int vqacl_set_gemm_sm_limit(int n) {
  g_sm_limit = n > 0 ? (n & ~1) : 0;   // even: the CTA-pair kernel launches clusters of two
  return 0;
}

template <int BN, bool A_MN, bool B_MN>
static int launch(const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& args, cudaStream_t stream) {
  using Cfg = GemmCfg<BN>;
  auto kern = gemm_bf16_tcgen05_kernel<BN, A_MN, B_MN>;
  static bool attr_set = false;
  if (!attr_set) {
    VQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int tiles = ((args.M + GEMM_BM - 1) / GEMM_BM) * ((args.N + BN - 1) / BN) * args.splits;
  const int grid = tiles < gemm_sms(args.sm_limit) ? tiles : gemm_sms(args.sm_limit);
  (void)vq_launch(kern, dim3(grid), dim3(GEMM_THREADS), Cfg::SMEM_BYTES, stream, ta, tb, args);
  VQ_LAUNCH_CHECK();
  return 0;
}

// Dynamic tile schedule of the CTA-pair kernel: a ring of {next item, pairs finished} counter pairs in device memory, one per
// launch in flight (the kernel's last pair resets its slot). VQACL_GEMM_DYN=0/1 overrides the default.
constexpr int SCHED_SLOTS = 256;
static uint32_t* g_sched = nullptr;
static int g_sched_next = 0;
static int g_dyn = [] { const char* e = getenv("VQACL_GEMM_DYN"); return e ? (e[0] == '1' ? 1 : 0) : 0; }();
extern "C" int vqacl_set_gemm_dynamic_schedule(int on) {
  g_dyn = on ? 1 : 0;
  return 0;
}

// CTA-pair kernel: clusters of 2 CTAs, 256 x 256 tiles (see gemm_tcgen05.cuh)
template <bool A_MN, bool B_MN>
static int launch_pair(const CUtensorMap& ta, const CUtensorMap& tb, const GemmArgs& args_in, cudaStream_t stream) {
  GemmArgs args = args_in;
  args.sched = nullptr;
  if (g_dyn && !args.tail) {
    if (!g_sched) {
      VQ_CUDA(cudaMalloc(&g_sched, SCHED_SLOTS * 2 * sizeof(uint32_t)));
      VQ_CUDA(cudaMemset(g_sched, 0, SCHED_SLOTS * 2 * sizeof(uint32_t)));
    }
    args.sched = g_sched + 2 * (g_sched_next++ % SCHED_SLOTS);
  }
  auto kern = gemm_bf16_tcgen05_2cta_kernel<A_MN, B_MN>;
  static bool attr_set = false;
  if (!attr_set) {
    VQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Gemm2Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int work = ((args.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM)) * ((args.N + GEMM2_BN - 1) / GEMM2_BN) * args.splits;
  const int max_pairs = gemm_sms(args.sm_limit) / 2;
  const int pairs = work < max_pairs ? work : max_pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = Gemm2Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = g_vq_pdl;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  VQ_CUDA(cudaLaunchKernelEx(&cfg, kern, ta, tb, args));
  ++g_vq_launches;
  return 0;
}

int gemm_bf16_grouped_mn(const GemmGroupProblem* probs, int n, int K, int epi, float alpha, int sm_limit, cudaStream_t stream) {
  VQ_CHECK(n >= 1 && n <= GEMM_GROUP_MAX, "gemm_grouped: %d problems (1..%d)", n, GEMM_GROUP_MAX);
  VQ_CHECK(epi == EPI_ATOMIC_F32 || epi == EPI_F32, "gemm_grouped: fp32 store / accumulate epilogues only");
  VQ_CHECK(K > 0, "gemm_grouped: empty contraction");
  (void)num_sms();
  VQ_CHECK(g_pair_enabled, "gemm_grouped: needs the CTA-pair kernel");
  GemmGroupMaps maps;
  GemmGroup grp{};
  grp.n = n;
  int total = 0;
  for (int i = 0; i < n; ++i) {
    const GemmGroupProblem& q = probs[i];
    VQ_CHECK(q.M > 0 && q.N > 0 && q.N % 8 == 0 && q.ldc % 8 == 0 && q.A && q.B && q.C, "gemm_grouped: bad problem %d (%d x %d)", i, q.M, q.N);
    if (make_tmap(&maps.a[i], q.A, q.M, K, q.lda, 64, GEMM_BK)) return 1;
    if (make_tmap(&maps.b[i], q.B, q.N, K, q.ldb, 64, GEMM_BK)) return 1;
    grp.M[i] = q.M; grp.N[i] = q.N; grp.ldc[i] = q.ldc; grp.C[i] = q.C;
    grp.tiles_n[i] = (q.N + GEMM2_BN - 1) / GEMM2_BN;
    grp.tile_start[i] = total;
    total += ((q.M + 2 * GEMM_BM - 1) / (2 * GEMM_BM)) * grp.tiles_n[i];
  }
  for (int i = n; i <= GEMM_GROUP_MAX; ++i) grp.tile_start[i] = total;
  for (int i = n; i < GEMM_GROUP_MAX; ++i) { maps.a[i] = maps.a[0]; maps.b[i] = maps.b[0]; }
  GemmArgs args{};
  args.epi = epi; args.K = K; args.alpha = alpha; args.splits = 1;
  args.M = probs[0].M; args.N = probs[0].N; args.C = probs[0].C; args.ldc = probs[0].ldc;   // unused by the grouped body
  auto kern = gemm_bf16_tcgen05_2cta_grouped_kernel<true, true>;
  static bool attr_set = false;
  if (!attr_set) {
    VQ_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Gemm2Cfg::SMEM_BYTES));
    attr_set = true;
  }
  const int max_pairs = gemm_sms(sm_limit) / 2;
  const int pairs = total < max_pairs ? total : max_pairs;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(GEMM_THREADS);
  cfg.dynamicSmemBytes = Gemm2Cfg::SMEM_BYTES;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = g_vq_pdl;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  VQ_CUDA(cudaLaunchKernelEx(&cfg, kern, maps, args, grp));
  ++g_vq_launches;
  return 0;
}

static int dispatch_pair(const GemmOperand& A, const GemmOperand& B, const GemmArgs& args, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (!A.mn_major) {
    if (make_tmap(&ta, A.ptr, args.K, args.M, A.ld, GEMM_BK, GEMM_BM)) return 1;
  } else {
    if (make_tmap(&ta, A.ptr, args.M, args.K, A.ld, 64, GEMM_BK)) return 1;
  }
  if (!B.mn_major) {
    if (make_tmap(&tb, B.ptr, args.K, args.N, B.ld, GEMM_BK, GEMM2_BN / 2)) return 1;   // each CTA loads half of the 256-wide B tile
  } else {
    if (make_tmap(&tb, B.ptr, args.N, args.K, B.ld, 64, GEMM_BK)) return 1;
  }
  if (!A.mn_major && !B.mn_major) return launch_pair<false, false>(ta, tb, args, stream);
  if (!A.mn_major && B.mn_major) return launch_pair<false, true>(ta, tb, args, stream);
  if (A.mn_major && B.mn_major) return launch_pair<true, true>(ta, tb, args, stream);
  VQ_CHECK(false, "gemm: A MN-major with B K-major is not instantiated");
}

template <int BN>
static int dispatch_major(const GemmOperand& A, const GemmOperand& B, const GemmArgs& args, cudaStream_t stream) {
  CUtensorMap ta, tb;
  if (!A.mn_major) {
    if (make_tmap(&ta, A.ptr, args.K, args.M, A.ld, GEMM_BK, GEMM_BM)) return 1;
  } else {
    if (make_tmap(&ta, A.ptr, args.M, args.K, A.ld, 64, GEMM_BK)) return 1;
  }
  if (!B.mn_major) {
    if (make_tmap(&tb, B.ptr, args.K, args.N, B.ld, GEMM_BK, BN)) return 1;
  } else {
    if (make_tmap(&tb, B.ptr, args.N, args.K, B.ld, 64, GEMM_BK)) return 1;
  }
  if (!A.mn_major && !B.mn_major) return launch<BN, false, false>(ta, tb, args, stream);
  if (!A.mn_major && B.mn_major) return launch<BN, false, true>(ta, tb, args, stream);
  if (A.mn_major && B.mn_major) return launch<BN, true, true>(ta, tb, args, stream);
  VQ_CHECK(false, "gemm: A MN-major with B K-major is not instantiated");
}

int gemm_split_count(int K, int splits) {
  const int kblocks = (K + GEMM_BK - 1) / GEMM_BK;
  if (splits < 1) splits = 1;
  if (splits > kblocks) splits = kblocks;
  const int per = (kblocks + splits - 1) / splits;   // k-blocks per split, rounded so that no split is empty
  return (kblocks + per - 1) / per;
}

int gemm_bf16(const GemmOperand& A, const GemmOperand& B, GemmArgs args, int force_bn, cudaStream_t stream) {
  VQ_CHECK(args.M > 0 && args.N > 0 && args.K > 0, "gemm: empty problem %d x %d x %d", args.M, args.N, args.K);
  VQ_CHECK(args.N % 8 == 0, "gemm: N=%d must be a multiple of 8", args.N);
  VQ_CHECK(args.ldc % 8 == 0 && args.ldc >= (args.epi == EPI_ARGMAX ? 1 : args.N), "gemm: ldc=%d must be a multiple of 8 and >= N=%d",
           args.ldc, args.N);
  // the epilogue stores (and the residual epilogue loads) 16-byte vectors; the mask epilogues access one u32 word per 32 columns
  VQ_CHECK(args.C && (args.epi == EPI_ARGMAX || (reinterpret_cast<uintptr_t>(args.C) & 15) == 0), "gemm: C %p is not 16-byte aligned", args.C);
  VQ_CHECK(args.epi != EPI_RESID_F32 || (args.R && (reinterpret_cast<uintptr_t>(args.R) & 15) == 0 && args.ldr % 4 == 0 && args.ldr >= args.N),
           "gemm: the residual epilogue needs a 16-byte aligned R with a pitch that is a multiple of 4 and >= N");
  VQ_CHECK(args.epi != EPI_RELUBWD_BF16 || args.R, "gemm: the ReLU-backward epilogue needs the sign bitmask R");
  VQ_CHECK((args.epi != EPI_RELU_BF16 && args.epi != EPI_RELUBWD_BF16) || !args.R || args.ldr >= (args.N + 31) / 32,
           "gemm: the sign bitmask needs ldr >= %d words", (args.N + 31) / 32);
  if (args.splits < 1) args.splits = 1;
  VQ_CHECK(args.splits == 1 || args.epi == EPI_ATOMIC_F32 || (args.epi == EPI_F32 && args.split_stride >= (long long)args.M * args.ldc),
           "gemm: split-K needs the atomic epilogue, or the fp32 one with a slab stride");
  if (args.splits == 1) args.split_stride = 0;
  if (args.tail) {
    VQ_CHECK((args.tail == 1 || args.tail == 2) && args.N == 768 && args.splits == 1 && (args.epi == EPI_RESID_F32 || args.epi == EPI_F32) &&
                 !A.mn_major && g_pair_enabled,
             "gemm: a row tail needs an fp32 768-wide output, no split-K and the CTA-pair kernel");
    VQ_CHECK(args.tail != 1 || (args.tail_w && args.tail_out && args.tail_ld % 4 == 0), "gemm: RMSNorm row tail: missing operands");
    VQ_CHECK(args.tail != 2 || (args.vt.boxes && args.vt.x && args.vt.N > 0), "gemm: VisualEmbedding row tail: missing operands");
    force_bn = 512;
  }
  if (args.epi == EPI_ARGMAX) {
    if (force_bn == 0) force_bn = args.M >= 192 ? 512 : 256;
    VQ_CHECK(force_bn == 256 || force_bn == 512, "gemm: the argmax epilogue needs 256-wide tiles");
    const int slots = (args.N + 255) / 256 * GEMM_EPI_GROUPS;
    VQ_CHECK(args.C && args.R && args.ldc >= slots && args.ldr >= slots, "gemm: argmax partial buffers need %d slots per row", slots);
  }
  const int kblocks = (args.K + GEMM_BK - 1) / GEMM_BK;
  args.splits = gemm_split_count(args.K, args.splits);
  int bn = force_bn;
  if (bn == 0) {
    // pick the tile shape that minimises waves x per-tile MMA time. Cycles per 64-deep k-block:
    //   128 x BN single-CTA tile: 4 MMAs, each bound by shared-memory traffic (TMA write + operand read) rather than the
    //   tensor pipe — 128 x 256 runs at 2/3 of the MMA rate (measured), the narrow tiles re-read A even more often;
    //   256 x 256 CTA-pair tile (bn = 512): 4 MMAs at the full rate on two SMs.
    const int tiles_m = (args.M + GEMM_BM - 1) / GEMM_BM;
    (void)num_sms();
    const int sms = gemm_sms(args.sm_limit);
    const int kb_split = (kblocks + args.splits - 1) / args.splits;
    const int cand[3] = {256, 128, 64};
    const int cyc[3] = {768, 400, 240};
    long best = -1;
    for (int i = 0; i < 3; ++i) {
      if (cand[i] > 64 && args.N < cand[i] / 2 + 8) continue;   // mostly-empty tile
      const long work = (long)tiles_m * ((args.N + cand[i] - 1) / cand[i]) * args.splits;
      const long waves = (work + sms - 1) / sms;
      const long cost = waves * ((long)kb_split * cyc[i] + 600 + cand[i] * 4);   // + pipeline fill and epilogue drain
      if (best < 0 || cost < best) { best = cost; bn = cand[i]; }
    }
    if (args.N >= 192 && args.M >= 192 && g_pair_enabled) {
      const long work = (long)((args.M + 255) / 256) * ((args.N + 255) / 256) * args.splits;
      const long waves = (work + sms / 2 - 1) / (sms / 2);
      const long cost = waves * ((long)kb_split * 512 + 900 + 1024);
      if (cost < best) { best = cost; bn = 512; }
    }
  }
  if (bn == 512) return dispatch_pair(A, B, args, stream);
  switch (bn) {
    case 256: return dispatch_major<256>(A, B, args, stream);
    case 128: return dispatch_major<128>(A, B, args, stream);
    case 64: return dispatch_major<64>(A, B, args, stream);
    default: VQ_CHECK(false, "gemm: unsupported BN %d", bn);
  }
}

}  // namespace vq

// ------------------------------------------------------------------------------------------
// C-ABI entry (see include/vqacl_b200.h)
// ------------------------------------------------------------------------------------------
/* grouped weight-gradient GEMM: problem i is C[i][M[i], N[i]] (+)= A[i]^T-stored [K, M[i]] x B[i] stored [K, N[i]] */
extern "C" int vqacl_gemm_bf16_grouped_mn(int n, const void* const* A, const int* lda, const void* const* B, const int* ldb, void* const* C,
                                          const int* ldc, const int* M, const int* N, int K, int epi, float alpha, void* stream) {
  VQ_CHECK(n >= 1 && n <= vq::GEMM_GROUP_MAX, "gemm_grouped: %d problems", n);
  vq::GemmGroupProblem pr[vq::GEMM_GROUP_MAX];
  for (int i = 0; i < n; ++i) pr[i] = vq::GemmGroupProblem{A[i], lda[i], B[i], ldb[i], C[i], ldc[i], M[i], N[i]};
  return vq::gemm_bf16_grouped_mn(pr, n, K, epi, alpha, 0, reinterpret_cast<cudaStream_t>(stream));
}

extern "C" int vqacl_gemm_bf16(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, void* C,
                               int ldc, const void* R, int ldr, int M, int N, int K, int epi, float alpha, int splits,
                               int force_bn, void* stream) {
  vq::GemmOperand a{A, lda, a_mn_major != 0}, b{B, ldb, b_mn_major != 0};
  vq::GemmArgs g{};
  g.epi = epi;
  g.M = M; g.N = N; g.K = K;
  g.C = C; g.ldc = ldc;
  g.R = R; g.ldr = ldr;
  g.alpha = alpha;
  g.splits = splits;
  return vq::gemm_bf16(a, b, g, force_bn, reinterpret_cast<cudaStream_t>(stream));
}

// split-K with one fp32 slab per split (the decoder FFN-out form, epilogue 5 with a slab stride)
extern "C" int vqacl_gemm_bf16_slabs(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, float* C, int ldc,
                                     long long split_stride, int M, int N, int K, float alpha, int splits, int force_bn, int* n_slabs,
                                     void* stream) {
  VQ_CHECK(n_slabs != nullptr, "gemm_slabs: n_slabs is null");
  vq::GemmOperand a{A, lda, a_mn_major != 0}, b{B, ldb, b_mn_major != 0};
  vq::GemmArgs g{};
  g.epi = vq::EPI_F32;
  g.M = M; g.N = N; g.K = K;
  g.C = C; g.ldc = ldc;
  g.alpha = alpha;
  g.splits = splits;
  g.split_stride = split_stride;
  if (vq::gemm_bf16(a, b, g, force_bn, reinterpret_cast<cudaStream_t>(stream))) return 1;
  *n_slabs = vq::gemm_split_count(K, splits);
  return 0;
}

// same with the epilogue dropout exposed (epi 1 and 2): drop_thr16 = round(p * 65536) (0 disables), drop_key = the per-launch
// 32-bit key; element (row, col) is kept iff the 16-bit lane ((row * N + col) & 1 ? hi : lo) of
// murmur3_fmix32(((row * N + col) >> 1) * 0x9E3779B1 + drop_key) is >= drop_thr16 and is then scaled by inv_keep
extern "C" int vqacl_gemm_bf16_ex(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, void* C,
                                  int ldc, const void* R, int ldr, int M, int N, int K, int epi, float alpha, int splits,
                                  int force_bn, uint32_t drop_thr16, float inv_keep, uint32_t drop_key, void* stream) {
  vq::GemmOperand a{A, lda, a_mn_major != 0}, b{B, ldb, b_mn_major != 0};
  vq::GemmArgs g{};
  g.epi = epi;
  g.M = M; g.N = N; g.K = K;
  g.C = C; g.ldc = ldc;
  g.R = R; g.ldr = ldr;
  g.alpha = alpha;
  g.splits = splits;
  g.drop_thr = drop_thr16; g.drop_inv_keep = inv_keep; g.seed = drop_key;
  return vq::gemm_bf16(a, b, g, force_bn, reinterpret_cast<cudaStream_t>(stream));
}

// nn.Linear + residual add + the T5LayerNorm that opens the next sub-layer, in one launch (HF T5LayerSelfAttention / T5LayerFF:
// hidden = hidden + dropout(layer(norm(hidden))) followed by the next layer_norm; hf5.5 modeling_t5.py:135-150, 347-377):
//   C(f32)[M,768] = R + A[M,K] * B[768,K]^T;   N_out(bf16)[M,768] = C * rsqrt(mean(C^2) + eps) * norm_w
// The norm runs as a row tail of the CTA-pair GEMM (see GemmArgs::tail).
extern "C" int vqacl_gemm_resid_rmsnorm(const void* A, int lda, const void* B, int ldb, float* C, const float* R, int M, int K,
                                        const float* norm_w, float eps, void* n_out_bf16, void* stream) {
  vq::GemmArgs g{};
  g.epi = vq::EPI_RESID_F32; g.M = M; g.N = 768; g.K = K; g.C = C; g.ldc = 768; g.R = R; g.ldr = 768; g.alpha = 1.f; g.splits = 1;
  g.tail = 1; g.tail_w = norm_w; g.tail_out = n_out_bf16; g.tail_ld = 768; g.tail_eps = eps;
  return vq::gemm_bf16(vq::GemmOperand{A, lda, false}, vq::GemmOperand{B, ldb, false}, g, 0, reinterpret_cast<cudaStream_t>(stream));
}

// VisualEmbedding.forward (modeling_t5_our.py:93-143) in one launch: feats(bf16)[B*N, F] @ Wf(bf16)[768, F]^T on tcgen05 with
// the rest of the module as the row tail (bias + RMSNorm, box projection + RMSNorm, order embeddings); featpre (fp32
// [B*N, 768]) receives the raw projection (the backward pass re-reads it); x [B, S, 768] rows [L, L + N) are written.
extern "C" int vqacl_visual_embed_fused(const void* feats_bf16, const void* Wf_bf16, int F, const float* boxes, const float* bf,
                                        const float* wf, const float* Wp, const float* bp, const float* wp, const float* img_emb,
                                        const float* shared, int V, int B, int N, int S, int L, float eps, float* featpre, float* x,
                                        void* stream) {
  vq::GemmArgs g{};
  g.epi = vq::EPI_F32; g.M = B * N; g.N = 768; g.K = F; g.C = featpre; g.ldc = 768; g.alpha = 1.f; g.splits = 1;
  g.tail = 2; g.tail_eps = eps;
  g.vt.boxes = boxes; g.vt.bf = bf; g.vt.wf = wf; g.vt.Wp = Wp; g.vt.bp = bp; g.vt.wp = wp; g.vt.img_emb = img_emb; g.vt.shared = shared;
  g.vt.x = x; g.vt.V = V; g.vt.N = N; g.vt.S = S; g.vt.L = L;
  return vq::gemm_bf16(vq::GemmOperand{feats_bf16, F, false}, vq::GemmOperand{Wf_bf16, F, false}, g, 0, reinterpret_cast<cudaStream_t>(stream));
}
