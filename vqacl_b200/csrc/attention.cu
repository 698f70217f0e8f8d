// Fused T5 attention for the VL-T5 shapes (S <= 64 keys/queries, d_kv = 64): the whole Q/K/V problem of one (batch, head)
// lives in shared memory (encoder forward: persistent 4-warp CTAs that stream the next problem in with cp.async while they work
// on the current one; encoder backward: one problem per 4-warp CTA; decoder self-attention: 4 single-warp problems per CTA;
// cross-attention: key-split across the 4 warps of a CTA). Output tiles leave through shared memory as full 128-byte rows.
// Scores are NOT scaled by 1/sqrt(d) (T5), the relative-position bias is read from the
// [num_buckets, H] embedding table through a host-precomputed rel->bucket map, and the additive masks of HF 4.2.1
// (-10000 key padding / causal, -1e9 cross) are applied in-kernel, so the [B,H,S,S] bias tensor the reference
// materialises (modeling_t5_our.py:258-273) never exists. Backward recomputes P from the saved log-sum-exp.
//
// Reference math: HF T5Attention (hf5.5 modeling_t5.py:277-338 == 4.2.1): softmax(QK^T + bias) V with dropout on P.
// The QK^T / PV cores are ~1 % of the step's FLOPs (SURVEY.md §8a5): they run on mma.sync m16n8k16 bf16 fragments;
// the tcgen05 path is reserved for the projections that carry the FLOPs.
#include "common.cuh"
#include "ops.h"

#include <string.h>

namespace vq {

constexpr int AT_S = 64;      // max queries / keys per problem
constexpr int AT_D = 64;      // head dim
constexpr int AT_P = 72;      // smem pitch (elements): 144 B rows -> conflict-free ldmatrix

VQ_DEVINL void ldsm_x4(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
VQ_DEVINL void ldsm_x4_t(uint32_t (&r)[4], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
VQ_DEVINL void ldsm_x2(uint32_t (&r)[2], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(smem_u32(p)));
}
VQ_DEVINL void ldsm_x2_t(uint32_t (&r)[2], const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0,%1}, [%2];" : "=r"(r[0]), "=r"(r[1]) : "r"(smem_u32(p)));
}
VQ_DEVINL void mma16816(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

typedef __nv_bfloat16 (*AttnTile)[AT_P];


// Load NM [rows<=64, 64] bf16 head slices into smem with 16-byte vectors. All global loads of a batch (4 per matrix and
// thread) are issued before the first shared store so that NM*4 requests per thread are in flight.
template <int NW, int NM>
VQ_DEVINL void load_heads(AttnTile const (&dst)[NM], const __nv_bfloat16* const (&src)[NM], const int (&ld)[NM], const int (&rows)[NM],
                          const int (&fill)[NM], int tid) {
  constexpr int T = NW * 32;
  int total[NM], maxtotal = 0;
#pragma unroll
  for (int m = 0; m < NM; ++m) {
    total[m] = fill[m] * (AT_D / 8);   // rows [rows, fill) are zero-filled: every tile row a consumer can touch is defined
    maxtotal = max(maxtotal, total[m]);
  }
  for (int base = 0; base < maxtotal; base += 4 * T) {
    uint4 v[NM][4];
#pragma unroll
    for (int m = 0; m < NM; ++m)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = base + u * T + tid;
        const int r = idx >> 3, c = (idx & 7) * 8;
        v[m][u] = make_uint4(0, 0, 0, 0);
        if (idx < total[m] && r < rows[m]) v[m][u] = *reinterpret_cast<const uint4*>(src[m] + (size_t)r * ld[m] + c);
      }
#pragma unroll
    for (int m = 0; m < NM; ++m)
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int idx = base + u * T + tid;
        if (idx < total[m]) *reinterpret_cast<uint4*>(&dst[m][idx >> 3][(idx & 7) * 8]) = v[m][u];
      }
  }
}

// ---- cp.async (LDGSTS) staging for the persistent, double-buffered encoder kernels: the tiles of problem i+1 stream into
//      the other shared-memory stage while the warps work on problem i; rows past the end of a matrix are zero-filled
//      by the copy itself (src-size 0).
VQ_DEVINL void cp_async16(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_u32(dst)), "l"(src), "r"(src_bytes) : "memory");
}
VQ_DEVINL void cp_async4(void* dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
VQ_DEVINL void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
VQ_DEVINL void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int NW, int NM>
VQ_DEVINL void load_heads_async(AttnTile const (&dst)[NM], const __nv_bfloat16* const (&src)[NM], const int (&ld)[NM], const int (&rows)[NM],
                                const int (&fill)[NM], int tid) {
  constexpr int T = NW * 32;
#pragma unroll
  for (int m = 0; m < NM; ++m) {
    const int total = fill[m] * (AT_D / 8);
    for (int idx = tid; idx < total; idx += T) {
      const int r = idx >> 3, c = (idx & 7) * 8;
      const bool ok = r < rows[m];
      cp_async16(&dst[m][r][c], ok ? src[m] + (size_t)r * ld[m] + c : src[m], ok ? 16 : 0);
    }
  }
}
// bias / key-mask header of a stage, asynchronously (gathers go through 4-byte cp.async, constants are plain stores: the
// stage is not being read by anyone while it is filled)
template <int NW>
VQ_DEVINL void load_bias_mask_async(float* sbias, float* skmask, const AttnArgs& p, const AttnBuckets& bk, int b, int h, int tid) {
  constexpr int T = NW * 32;
  if (p.rel_mode) {
    for (int r = tid; r < 2 * AT_S - 1; r += T) cp_async4(&sbias[r], &p.rel_table[(int)bk.b[r] * p.H + h]);
  }
  for (int j = tid; j < AT_S; j += T) {
    if (j < p.Sk && p.keymask) cp_async4(&skmask[j], &p.keymask[(size_t)b * p.Sk + j]);
    else skmask[j] = j < p.Sk ? 0.f : -INFINITY;
  }
}

// A fragment (m16 x k16) of row-major X[m][k] at (m0, k0)
VQ_DEVINL void frag_a(uint32_t (&a)[4], const __nv_bfloat16 (*X)[AT_P], int m0, int k0, int lane) {
  const int mi = lane >> 3, r = lane & 7;
  ldsm_x4(a, &X[m0 + (mi & 1) * 8 + r][k0 + (mi >> 1) * 8]);
}
// A fragment of X^T where X is stored [k][m] row-major
VQ_DEVINL void frag_a_t(uint32_t (&a)[4], const __nv_bfloat16 (*X)[AT_P], int m0, int k0, int lane) {
  const int mi = lane >> 3, r = lane & 7;
  ldsm_x4_t(a, &X[k0 + (mi >> 1) * 8 + r][m0 + (mi & 1) * 8]);
}
// B fragment (k16 x n8) where B[k][n] is stored as X[n][k] row-major
VQ_DEVINL void frag_b(uint32_t (&b)[2], const __nv_bfloat16 (*X)[AT_P], int n0, int k0, int lane) {
  const int l = lane & 15, mi = l >> 3, r = l & 7;
  ldsm_x2(b, &X[n0 + r][k0 + mi * 8]);
}
// B fragment where B[k][n] is stored as X[k][n] row-major
VQ_DEVINL void frag_b_t(uint32_t (&b)[2], const __nv_bfloat16 (*X)[AT_P], int n0, int k0, int lane) {
  const int l = lane & 15, mi = l >> 3, r = l & 7;
  ldsm_x2_t(b, &X[k0 + mi * 8 + r][n0]);
}

// Write a warp's [16 x 64] tile (m16n8 accumulator layout: rows m0 + g and m0 + g + 8, columns nt * 8 + 2t) to global memory
// as full 128-byte rows: the tile is first packed into rows [m0, m0 + 16) of a shared tile that only this warp touches any
// more, then each quarter-warp moves one row with 16-byte vectors (4-byte stores straight from the fragments cover only half
// of every 32-byte sector per instruction and keep the LSU busy long after the math is done).
VQ_DEVINL void store_tile16(AttnTile stg, int m0, const float (&acc)[8][4], __nv_bfloat16* gbase, int ld, int nrows, int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int r = 0; r < 2; ++r)
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) *reinterpret_cast<uint32_t*>(&stg[m0 + g + r * 8][nt * 8 + 2 * t]) = pack_bf16(acc[nt][2 * r], acc[nt][2 * r + 1]);
  __syncwarp();
#pragma unroll
  for (int it = 0; it < 4; ++it) {
    const int row = m0 + it * 4 + (lane >> 3), c = (lane & 7) * 8;
    if (row < nrows) *reinterpret_cast<uint4*>(gbase + (size_t)row * ld + c) = *reinterpret_cast<const uint4*>(&stg[row][c]);
  }
  __syncwarp();
}


// Shared memory is carved per launch for the rows that exist (rounded up to 16), and the CTA has one warp per 16 query
// rows (backward: per 16 query or key rows), so the decoder's tiny problems (Sq = T <= 10) run as 1-warp CTAs with 7-21 KB
// of smem and many CTAs per SM instead of idling three warps and 28-56 KB.
constexpr int AT_HDR_BYTES = (2 * AT_S + AT_S + 64) * 4;   // bias[128] | kmask[64] | dbucket[64] (floats)
VQ_DEVINL int rows16(int n) { return (n + 15) & ~15; }
// query-side tiles hold round_up(Sq, 16) rows, key-side tiles NKT * 8 rows (16 or 64)
static inline int attn_smem_fwd(int Sq, int krows) { return AT_HDR_BYTES + (((Sq + 15) & ~15) + 2 * krows) * AT_P * 2; }
static inline int attn_smem_bwd(int Sq, int krows) { return AT_HDR_BYTES + (4 * ((Sq + 15) & ~15) + 2 * krows) * AT_P * 2; }

// two adjacent B fragments (k16 x n16) at once; B[k][n] stored as X[n][k] row-major: regs {b(n0)[0], b(n0)[1], b(n0+8)[0], b(n0+8)[1]}
VQ_DEVINL void frag_b2(uint32_t (&b)[4], const __nv_bfloat16 (*X)[AT_P], int n0, int k0, int lane) {
  const int mi = lane >> 3, r = lane & 7;
  ldsm_x4(b, &X[n0 + (mi >> 1) * 8 + r][k0 + (mi & 1) * 8]);
}
// same for B[k][n] stored as X[k][n] row-major
VQ_DEVINL void frag_b2_t(uint32_t (&b)[4], const __nv_bfloat16 (*X)[AT_P], int n0, int k0, int lane) {
  const int mi = lane >> 3, r = lane & 7;
  ldsm_x4_t(b, &X[k0 + (mi & 1) * 8 + r][n0 + (mi >> 1) * 8]);
}
VQ_DEVINL void mma2(float (&d0)[4], float (&d1)[4], const uint32_t (&a)[4], const uint32_t (&b)[4]) {
  const uint32_t b0[2] = {b[0], b[1]}, b1[2] = {b[2], b[3]};
  mma16816(d0, a, b0);
  mma16816(d1, a, b1);
}

// scores for the warp's 16 query rows vs NKT key tiles of 8 (NKT = 2: decoder self-attention, Sk <= 16; NKT = 8: up to
// 64 keys), bias/mask applied; keys >= Sk get -inf. The additive terms are organised so that the common case costs one
// FADD per score: the key-side term (padding mask, -inf beyond Sk) comes from smem as float2, the relative-position bias
// is only visited for the tiles that intersect the biased region (encoder: the text x text corner), the causal term only
// for decoder self-attention.
template <int NKT>
VQ_DEVINL void scores_tile(float (&s)[NKT][4], const __nv_bfloat16 (*sq)[AT_P], const __nv_bfloat16 (*sk)[AT_P],
                           const float* sbias, const float* skmask, const AttnArgs& p, int m0, int lane) {
#pragma unroll
  for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) s[nt][i] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a[4];
    frag_a(a, sq, m0, kk * 16, lane);
#pragma unroll
    for (int nt = 0; nt < NKT; nt += 2) {
      uint32_t b[4];
      frag_b2(b, sk, nt * 8, kk * 16, lane);
      mma2(s[nt], s[nt + 1], a, b);
    }
  }
  const int g = lane >> 2, t = lane & 3;
  // key-side term: skmask[] already holds -inf for keys >= Sk (load_bias_mask)
#pragma unroll
  for (int nt = 0; nt < NKT; ++nt) {
    const float2 ka = *reinterpret_cast<const float2*>(skmask + nt * 8 + 2 * t);
    s[nt][0] += ka.x; s[nt][1] += ka.y; s[nt][2] += ka.x; s[nt][3] += ka.y;
  }
  const int q0 = m0 + g + p.q_off;   // absolute position of this thread's first query row (second is q0 + 8)
  if (p.rel_mode == 2) {
    // bias everywhere (decoder self-attention); rel = key - query is within +-63 for every row that exists (check_args:
    // q_off + Sq <= 64). Padded rows (>= Sq, never stored) take the last row's position, so that with a query offset (KV-cache
    // decoding) their bias index does not leave [0, 127) either.
    const float* bp0 = sbias + (2 * t - (min(m0 + g, p.Sq - 1) + p.q_off) + (AT_S - 1));
    const float* bp1 = sbias + (2 * t - (min(m0 + g + 8, p.Sq - 1) + p.q_off) + (AT_S - 1));
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt) {
      s[nt][0] += bp0[nt * 8]; s[nt][1] += bp0[nt * 8 + 1]; s[nt][2] += bp1[nt * 8]; s[nt][3] += bp1[nt * 8 + 1];
    }
  } else if (p.rel_mode == 1 && m0 < p.Lt) {
    // bias on the text x text corner only (encoder): rows / key tiles beyond Lt are skipped warp-uniformly
    const bool r0 = q0 < p.Lt, r1 = q0 + 8 < p.Lt;
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt)
      if (nt * 8 < p.Lt) {
        const int kj = nt * 8 + 2 * t;
        const float* bp = sbias + (kj - q0 + (AT_S - 1));
        const bool c0 = kj < p.Lt, c1 = kj + 1 < p.Lt;
        if (r0 && c0) s[nt][0] += bp[0];
        if (r0 && c1) s[nt][1] += bp[1];
        if (r1 && c0) s[nt][2] += bp[-8];
        if (r1 && c1) s[nt][3] += bp[-7];
      }
  }
  if (p.causal) {
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt) {
      const int kj = nt * 8 + 2 * t;
      if (kj > q0) s[nt][0] += -10000.0f;
      if (kj + 1 > q0) s[nt][1] += -10000.0f;
      if (kj > q0 + 8) s[nt][2] += -10000.0f;
      if (kj + 1 > q0 + 8) s[nt][3] += -10000.0f;
    }
  }
}

// Bias / key-mask header of a problem in two halves: `fetch` issues every global load into registers, `store` writes them to
// shared memory. The tile loads go BETWEEN the two: a gather that feeds a shared store directly (the single-function form this
// replaces) stalls the thread for one memory round trip per loop iteration — with one warp per problem that was 6 dependent
// round trips before the first tile load was even issued (ncu: stall_long_sb on every STS of the header).
template <int NW>
struct BiasMaskRegs {
  static constexpr int T = NW * 32, NB = (2 * AT_S + T - 1) / T, NK = (AT_S + T - 1) / T;
  float bias[NB], kmask[NK];
  VQ_DEVINL void fetch(const AttnArgs& p, const AttnBuckets& bk, int b, int h, int tid) {
#pragma unroll
    for (int it = 0; it < NB; ++it) {
      const int r = it * T + tid;
      bias[it] = (p.rel_mode && r < 2 * AT_S - 1) ? p.rel_table[(int)bk.b[r] * p.H + h] : 0.f;
    }
    // key-side additive term: padding mask for existing keys, -inf beyond Sk
#pragma unroll
    for (int it = 0; it < NK; ++it) {
      const int j = it * T + tid;
      kmask[it] = j < p.Sk ? (p.keymask ? p.keymask[(size_t)b * p.Sk + j] : 0.f) : -INFINITY;
    }
  }
  VQ_DEVINL void store(float* sbias, float* skmask, const AttnArgs& p, int tid) const {
    if (p.rel_mode) {
#pragma unroll
      for (int it = 0; it < NB; ++it) {
        const int r = it * T + tid;
        if (r < 2 * AT_S - 1) sbias[r] = bias[it];
      }
    }
#pragma unroll
    for (int it = 0; it < NK; ++it) {
      const int j = it * T + tid;
      if (j < AT_S) skmask[j] = kmask[it];
    }
  }
};

struct AttnSmemF { float* bias; float* kmask; AttnTile q, k, v; };
VQ_DEVINL AttnSmemF attn_carve_fwd(uint8_t* raw, int qrows, int krows) {
  AttnSmemF sm;
  sm.bias = reinterpret_cast<float*>(raw);
  sm.kmask = sm.bias + 2 * AT_S;
  sm.q = reinterpret_cast<AttnTile>(raw + AT_HDR_BYTES);
  sm.k = sm.q + qrows;
  sm.v = sm.k + krows;
  return sm;
}

// scores -> softmax (+ dropout) -> O = P V for the 16 query rows of one warp; the tiles of problem vblk = b * H + h are in sm
template <int NW, int NKT>
VQ_DEVINL void attn_fwd_compute(const AttnArgs& p, const AttnSmemF& sm, int vblk, int b, int h, int warp, int lane) {
  const int m0 = warp * 16;
  if (m0 >= p.Sq) return;
  float s[NKT][4];
  scores_tile<NKT>(s, sm.q, sm.k, sm.bias, sm.kmask, p, m0, lane);
  const int g = lane >> 2, t = lane & 3;
  // row-wise softmax (rows g and g+8 of this warp's tile), fp32
  float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) mx[i >> 1] = fmaxf(mx[i >> 1], s[nt][i]);
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
  }
  float sum[2] = {0.f, 0.f};
#pragma unroll
  for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float e = __expf(s[nt][i] - mx[i >> 1]);
      s[nt][i] = e;
      sum[i >> 1] += e;
    }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
  }
  const float inv[2] = {1.f / sum[0], 1.f / sum[1]};
  if (t == 0 && p.lse) {
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = m0 + g + r * 8;
      if (qi < p.Sq) p.lse[((size_t)b * p.H + h) * p.Sq + qi] = mx[r] + __logf(sum[r]);
    }
  }
#pragma unroll
  for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float s0 = inv[r], s1 = inv[r];
      if (p.drop_thr) {
        float d0, d1;
        vq_dropout_pair(p.seed, attn_pair_idx(vblk, m0 + g + r * 8, nt * 8 + 2 * t), p.drop_thr, p.drop_inv_keep, d0, d1);
        s0 *= d0; s1 *= d1;
      }
      s[nt][2 * r] *= s0;
      s[nt][2 * r + 1] *= s1;
    }
  // O = P V
  float o[8][4];
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) o[nt][i] = 0.f;
#pragma unroll
  for (int kk = 0; kk < NKT / 2; ++kk) {
    uint32_t a[4];
    a[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
    a[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
    a[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
    a[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
    for (int nt = 0; nt < 8; nt += 2) {
      uint32_t bb[4];
      frag_b2_t(bb, sm.v, nt * 8, kk * 16, lane);
      mma2(o[nt], o[nt + 1], a, bb);
    }
  }
  // this warp's rows of the q tile are dead after the scores: stage O there
  store_tile16(sm.q, m0, o, p.o + (size_t)b * (p.o_bstride ? p.o_bstride : (long long)p.Sq * p.ldo) + h * AT_D, p.ldo, p.Sq, lane);
}

// HPC > 1 (only with NW == 1): the CTA holds HPC independent single-warp problems (consecutive (batch, head) pairs), each
// with its own smem slice — the decoder's 3840 tiny problems are otherwise bound by the CTA dispatch rate.
// NW == 4 (encoder-sized problems): persistent CTAs, each walks over problems blockIdx.x, blockIdx.x + gridDim.x, ... with
// two shared-memory stages; the cp.async copies of the next problem are in flight while the current one is computed, so
// HBM stays busy during the math instead of only between CTA launches.
template <int NW, int NKT, int HPC>
__global__ void __launch_bounds__(NW * 32 * HPC, NW == 4 ? 3 : 16 / (NW * HPC)) attn_fwd_kernel(const AttnArgs p, const __grid_constant__ AttnBuckets bk) {
  static_assert(HPC == 1 || NW == 1, "several problems per CTA only for single-warp problems");
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  if constexpr (NW == 4) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nprob = p.B * p.H;
    const int stage_bytes = AT_HDR_BYTES + (rows16(p.Sq) + 2 * NKT * 8) * AT_P * 2;
    auto issue = [&](int vb, int stage) {
      const AttnSmemF sm = attn_carve_fwd(at_smem_base + stage * stage_bytes, rows16(p.Sq), NKT * 8);
      const int b = vb / p.H, h = vb % p.H;
      const AttnTile dst[3] = {sm.q, sm.k, sm.v};
      const __nv_bfloat16* const src[3] = {p.q + (size_t)b * (p.q_bstride ? p.q_bstride : (long long)p.Sq * p.ldq) + h * AT_D,
                                           p.k + (size_t)b * (p.k_bstride ? p.k_bstride : (long long)p.Sk * p.ldk) + h * AT_D,
                                           p.v + (size_t)b * (p.v_bstride ? p.v_bstride : (long long)p.Sk * p.ldv) + h * AT_D};
      const int ld[3] = {p.ldq, p.ldk, p.ldv};
      const int rows[3] = {p.Sq, p.Sk, p.Sk};
      const int fill[3] = {rows16(p.Sq), NKT * 8, NKT * 8};
      load_bias_mask_async<NW>(sm.bias, sm.kmask, p, bk, b, h, tid);
      load_heads_async<NW, 3>(dst, src, ld, rows, fill, tid);
    };
    int vblk = blockIdx.x, stage = 0;
    if (vblk < nprob) issue(vblk, 0);
    cp_async_commit();
    for (; vblk < nprob; vblk += gridDim.x) {
      if (vblk + (int)gridDim.x < nprob) issue(vblk + gridDim.x, stage ^ 1);
      cp_async_commit();
      cp_async_wait<1>();        // everything but the copies just issued has landed: this problem's stage is complete
      __syncthreads();
      const AttnSmemF sm = attn_carve_fwd(at_smem_base + stage * stage_bytes, rows16(p.Sq), NKT * 8);
      attn_fwd_compute<NW, NKT>(p, sm, vblk, vblk / p.H, vblk % p.H, warp, lane);
      __syncthreads();           // all warps are done with this stage before the next-but-one problem is copied into it
      stage ^= 1;
    }
  } else {
    const int vblk = HPC == 1 ? (int)blockIdx.x : (int)blockIdx.x * HPC + (int)(threadIdx.x >> 5);   // problem index = b * H + h
    if (vblk >= p.B * p.H) return;
    const int tid = HPC == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    uint8_t* at_smem_raw = at_smem_base + (HPC == 1 ? 0 : (threadIdx.x >> 5) * (AT_HDR_BYTES + (rows16(p.Sq) + 2 * NKT * 8) * AT_P * 2));
    const AttnSmemF sm = attn_carve_fwd(at_smem_raw, rows16(p.Sq), NKT * 8);
    const int b = vblk / p.H, h = vblk % p.H;
    const int warp = tid >> 5, lane = tid & 31;
    {
      const AttnTile dst[3] = {sm.q, sm.k, sm.v};
      const __nv_bfloat16* const src[3] = {p.q + (size_t)b * (p.q_bstride ? p.q_bstride : (long long)p.Sq * p.ldq) + h * AT_D,
                                           p.k + (size_t)b * (p.k_bstride ? p.k_bstride : (long long)p.Sk * p.ldk) + h * AT_D,
                                           p.v + (size_t)b * (p.v_bstride ? p.v_bstride : (long long)p.Sk * p.ldv) + h * AT_D};
      const int ld[3] = {p.ldq, p.ldk, p.ldv};
      const int rows[3] = {p.Sq, p.Sk, p.Sk};
      const int fill[3] = {rows16(p.Sq), NKT * 8, NKT * 8};
      BiasMaskRegs<NW> hdr;
      hdr.fetch(p, bk, b, h, tid);
      load_heads<NW, 3>(dst, src, ld, rows, fill, tid);
      hdr.store(sm.bias, sm.kmask, p, tid);
    }
    if (NW == 1) __syncwarp(); else __syncthreads();
    attn_fwd_compute<NW, NKT>(p, sm, vblk, b, h, warp, lane);
  }
}

struct AttnSmemB { float* bias; float* kmask; float* dbucket; AttnTile q, dO, P, dS, k, v; };

// backward of one problem whose q / dO / k / v tiles (and bias header, zeroed dbucket) are in sm; P and dS are scratch tiles
// lse_pre: the saved log-sum-exp of this lane's two query rows (rows m0 + g and m0 + g + 8 of its warp's block; +inf beyond
// Sq), fetched by the caller together with the tile loads so that no global round trip sits in the middle of the math
template <int NW, int NKT>
VQ_DEVINL void attn_bwd_compute(const AttnArgs& p, const AttnBuckets& bk, const AttnSmemB& sm, int vblk, int b, int h, int tid,
                                const float (&lse_pre)[2]) {
  const int warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t = lane & 3;
  const int nqk = (p.Sq + 15) >> 4;   // query blocks of 16
  // ---- phase 1: this warp owns 16 query rows (warps past the last query block only take part in phase 2) ----
  const int m0 = warp * 16;
  if (m0 < p.Sq) {
    float s[NKT][4];
    scores_tile<NKT>(s, sm.q, sm.k, sm.bias, sm.kmask, p, m0, lane);
    const float lse[2] = {lse_pre[0], lse_pre[1]};                               // rows >= Sq: +inf -> P = 0
    // dPd = dO V^T
    float dp[NKT][4];
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) dp[nt][i] = 0.f;
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      uint32_t a[4];
      frag_a(a, sm.dO, m0, kk * 16, lane);
#pragma unroll
      for (int nt = 0; nt < NKT; nt += 2) {
        uint32_t bb[4];
        frag_b2(bb, sm.v, nt * 8, kk * 16, lane);
        mma2(dp[nt], dp[nt + 1], a, bb);
      }
    }
    float dsum[2] = {0.f, 0.f};
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int qi = m0 + g + r * 8, kj = nt * 8 + 2 * t;
        float sc0 = 1.f, sc1 = 1.f;
        if (p.drop_thr) vq_dropout_pair(p.seed, attn_pair_idx(vblk, qi, kj), p.drop_thr, p.drop_inv_keep, sc0, sc1);
        const float p0 = __expf(s[nt][2 * r] - lse[r]), p1 = __expf(s[nt][2 * r + 1] - lse[r]);  // exp(-inf) = 0: masked keys / padded rows
        const float d0 = dp[nt][2 * r] * sc0, d1 = dp[nt][2 * r + 1] * sc1;                          // dP
        s[nt][2 * r] = p0; s[nt][2 * r + 1] = p1;
        dp[nt][2 * r] = d0; dp[nt][2 * r + 1] = d1;
        dsum[r] += p0 * d0 + p1 * d1;
        *reinterpret_cast<uint32_t*>(&sm.P[qi][kj]) = pack_bf16(p0 * sc0, p1 * sc1);                  // dropped P, for dV
      }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      dsum[r] += __shfl_xor_sync(0xffffffffu, dsum[r], 1);
      dsum[r] += __shfl_xor_sync(0xffffffffu, dsum[r], 2);
    }
#pragma unroll
    for (int nt = 0; nt < NKT; ++nt)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const float ds0 = s[nt][2 * r] * (dp[nt][2 * r] - dsum[r]), ds1 = s[nt][2 * r + 1] * (dp[nt][2 * r + 1] - dsum[r]);
        s[nt][2 * r] = ds0; s[nt][2 * r + 1] = ds1;
        *reinterpret_cast<uint32_t*>(&sm.dS[m0 + g + r * 8][nt * 8 + 2 * t]) = pack_bf16(ds0, ds1);
      }
    // dQ = dS K   (B[k=key][n=d] stored [key][d] -> transposed fragment loads)
    float dq[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) dq[nt][i] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NKT / 2; ++kk) {
      uint32_t a[4];
      a[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
      a[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
      a[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
      a[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
      for (int nt = 0; nt < 8; nt += 2) {
        uint32_t bb[4];
        frag_b2_t(bb, sm.k, nt * 8, kk * 16, lane);
        mma2(dq[nt], dq[nt + 1], a, bb);
      }
    }
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = m0 + g + r * 8;
      if (qi < p.Sq) {
        __nv_bfloat16* dst = p.dq + ((size_t)b * p.Sq + qi) * p.lddq + h * AT_D + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf16(dq[nt][2 * r], dq[nt][2 * r + 1]);
      }
    }
  }
  if (NW == 1) __syncwarp(); else __syncthreads();
  // ---- relative-position-bias gradient: d table[bucket(k - q)] += dS[q][k]; one thread per diagonal of the biased
  //      region sums its <= 64 entries from smem, then one smem atomic per diagonal and one global atomic per bucket.
  //      Without a bias (rel_mode 0) there is no region and the table is left alone. ----
  const bool d_bias = p.d_rel_table && p.rel_mode;
  if (d_bias) {
    const int nq = p.rel_mode == 1 ? min(p.Sq, p.Lt) : p.Sq;
    const int nk = p.rel_mode == 1 ? min(p.Sk, p.Lt) : p.Sk;
    const int ndiag = nq + nk - 1;
    const int parts = min(4, max(1, (NW * 32) / ndiag));   // split every diagonal over up to 4 threads: the loop is latency-bound
    for (int wi = tid; wi < ndiag * parts; wi += NW * 32) {
      const int dgi = wi / parts, part = wi - dgi * parts;
      const int rel = dgi - (nq - 1);   // k - q
      const int q_lo = max(0, -rel), len = min(nq, nk - rel) - q_lo;
      const int qa = q_lo + len * part / parts, qb = q_lo + len * (part + 1) / parts;
      float acc = 0.f;
      for (int qi = qa; qi < qb; ++qi) acc += __bfloat162float(sm.dS[qi][qi + rel]);
      if (qb > qa) atomicAdd(&sm.dbucket[(int)bk.b[rel + (AT_S - 1)]], acc);
    }
  }
  // ---- phase 2: this warp owns 16 key rows: dV = Pd^T dO, dK = dS^T Q (contraction over the query blocks that exist) ----
  if (m0 < p.Sk) {
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[nt][i] = dk[nt][i] = 0.f;
#pragma unroll
    for (int kk = 0; kk < NW; ++kk) {
      if (kk < nqk) {
        uint32_t ap[4], as[4];
        frag_a_t(ap, sm.P, m0, kk * 16, lane);
        frag_a_t(as, sm.dS, m0, kk * 16, lane);
#pragma unroll
        for (int nt = 0; nt < 8; nt += 2) {
          uint32_t b1[4], b2[4];
          frag_b2_t(b1, sm.dO, nt * 8, kk * 16, lane);
          frag_b2_t(b2, sm.q, nt * 8, kk * 16, lane);
          mma2(dv[nt], dv[nt + 1], ap, b1);
          mma2(dk[nt], dk[nt + 1], as, b2);
        }
      }
    }
    // the k / v tiles are dead since the end of phase 1: stage this warp's 16 rows of dK / dV in them
    store_tile16(sm.k, m0, dk, p.dk + (size_t)b * p.Sk * p.lddk + h * AT_D, p.lddk, p.Sk, lane);
    store_tile16(sm.v, m0, dv, p.dv + (size_t)b * p.Sk * p.lddv + h * AT_D, p.lddv, p.Sk, lane);
  }
  if (d_bias) {
    if (NW == 1) __syncwarp(); else __syncthreads();
    for (int i = tid; i < 64; i += NW * 32) {
      const float v = sm.dbucket[i];
      if (v != 0.f) atomicAdd(&p.d_rel_table[i * p.H + h], v);
    }
  }
}

template <int NW, int NKT, int HPC>
__global__ void __launch_bounds__(NW * 32 * HPC, NW == 4 ? 4 : 8 / HPC) attn_bwd_kernel(const AttnArgs p, const __grid_constant__ AttnBuckets bk) {
  static_assert(HPC == 1 || NW == 1, "several problems per CTA only for single-warp problems");
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  // (a persistent double-buffered variant like the forward kernel's was measured slower here: its 93 KB of shared memory
  //  allow 2 CTAs = 8 warps per SM, and the backward math needs more resident warps than that to hide its own latency)
  {
    const int vblk = HPC == 1 ? (int)blockIdx.x : (int)blockIdx.x * HPC + (int)(threadIdx.x >> 5);   // problem index = b * H + h
    if (vblk >= p.B * p.H) return;
    const int tid = HPC == 1 ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    uint8_t* at_smem_raw = at_smem_base + (HPC == 1 ? 0 : (threadIdx.x >> 5) * (AT_HDR_BYTES + (4 * rows16(p.Sq) + 2 * NKT * 8) * AT_P * 2));
    AttnSmemB sm;
    sm.bias = reinterpret_cast<float*>(at_smem_raw);
    sm.kmask = sm.bias + 2 * AT_S;
    sm.dbucket = sm.kmask + AT_S;
    sm.q = reinterpret_cast<AttnTile>(at_smem_raw + AT_HDR_BYTES);
    sm.dO = sm.q + rows16(p.Sq);
    sm.P = sm.dO + rows16(p.Sq);
    sm.dS = sm.P + rows16(p.Sq);
    sm.k = sm.dS + rows16(p.Sq);
    sm.v = sm.k + NKT * 8;
    const int b = vblk / p.H, h = vblk % p.H;
    float lse_pre[2];
    {
      const AttnTile dst[4] = {sm.q, sm.k, sm.v, sm.dO};
      const __nv_bfloat16* const src[4] = {p.q + (size_t)b * p.Sq * p.ldq + h * AT_D, p.k + (size_t)b * p.Sk * p.ldk + h * AT_D,
                                           p.v + (size_t)b * p.Sk * p.ldv + h * AT_D, p.dO + (size_t)b * p.Sq * p.ldo + h * AT_D};
      const int ld[4] = {p.ldq, p.ldk, p.ldv, p.ldo};
      const int rows[4] = {p.Sq, p.Sk, p.Sk, p.Sq};
      const int fill[4] = {rows16(p.Sq), NKT * 8, NKT * 8, rows16(p.Sq)};
      BiasMaskRegs<NW> hdr;
      hdr.fetch(p, bk, b, h, tid);
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int qi = (tid >> 5) * 16 + ((tid & 31) >> 2) + r * 8;
        lse_pre[r] = qi < p.Sq ? p.lse[((size_t)b * p.H + h) * p.Sq + qi] : INFINITY;
      }
      load_heads<NW, 4>(dst, src, ld, rows, fill, tid);
      hdr.store(sm.bias, sm.kmask, p, tid);
    }
    for (int i = tid; i < 64; i += NW * 32) sm.dbucket[i] = 0.f;
    if (NW == 1) __syncwarp(); else __syncthreads();
    attn_bwd_compute<NW, NKT>(p, bk, sm, vblk, b, h, tid, lse_pre);
  }
}

// =====================================================================================================================
// Key-split kernels for few queries against many keys (decoder cross-attention: Sq = T <= 16 queries, 58 keys).
// One CTA per (batch, head), 4 warps, warp w owns keys [16w, 16w+16). With one 16-row query tile the generic kernel would
// leave three warps idle; here every warp runs a complete softmax over its 16 keys (2 key tiles) and the per-warp results
// (row maximum, sum, partial P.V; backward: partial dS.K) are parked in shared memory and merged after one barrier
// (profiles/r01_summary.md: the shared fp32 atomics this replaced were 28 % of the kernel's stall samples).
// Backward needs no cross-warp softmax statistic: P = exp(S - lse) from the saved log-sum-exp and
// D = rowsum(dO * O) from the saved output (also valid with dropout: O was produced by the dropped probabilities).
// =====================================================================================================================
constexpr int KS_WARPS = 4;
constexpr int KS_OP = 68;   // pitch (floats) of the fp32 [16][64] accumulator tile: conflict-light for the fragment layout
struct KsSmemFwd {
  __nv_bfloat16 q[16][AT_P], k[AT_S][AT_P], v[AT_S][AT_P];
  float kmask[AT_S];
  float pm[KS_WARPS][16], pl[KS_WARPS][16];
};
// fp32 partial [16 queries x 64] tile of warp w, parked in shared memory the warp owns and no longer needs: query rows 0-7 in
// its 16 rows of the k tile, rows 8-15 in its 16 rows of the v tile (8 x KS_OP floats = 2176 B <= 16 x 144 B)
VQ_DEVINL float* ks_partial_row(__nv_bfloat16 (*k)[AT_P], __nv_bfloat16 (*v)[AT_P], int w, int qi) {
  return reinterpret_cast<float*>(qi < 8 ? &k[16 * w][0] : &v[16 * w][0]) + (qi & 7) * KS_OP;
}

// Every warp runs a complete softmax over ITS 16 keys (own maximum m_w, own sum l_w, un-normalised partial O_w = P_w V_w) and
// parks the partial in shared memory; the partials are merged flash-decoding style, O = sum_w e^(m_w - M) O_w / sum_w e^(m_w - M) l_w
// with M = max_w m_w: one barrier after the loads and one before the merge, no shared atomics (fp32 shared atomicAdd is a CAS loop).
__global__ void __launch_bounds__(KS_WARPS * 32, 8) attn_ks_fwd_kernel(const AttnArgs p) {
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  KsSmemFwd& sm = *reinterpret_cast<KsSmemFwd*>(at_smem_base);
  const int vblk = blockIdx.x, b = vblk / p.H, h = vblk % p.H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  {
    const AttnTile dst[3] = {sm.q, sm.k, sm.v};
    const __nv_bfloat16* const src[3] = {p.q + (size_t)b * (p.q_bstride ? p.q_bstride : (long long)p.Sq * p.ldq) + h * AT_D,
                                         p.k + (size_t)b * (p.k_bstride ? p.k_bstride : (long long)p.Sk * p.ldk) + h * AT_D,
                                         p.v + (size_t)b * (p.v_bstride ? p.v_bstride : (long long)p.Sk * p.ldv) + h * AT_D};
    const int ld[3] = {p.ldq, p.ldk, p.ldv};
    const int rows[3] = {p.Sq, p.Sk, p.Sk};
    const int fill[3] = {16, AT_S, AT_S};
    // the key-mask value is loaded into a register first and stored after the tile loads have been issued: a load feeding a
    // shared store directly would stall this thread for a DRAM round trip before its tile loads even start
    float kmv = -INFINITY;
    if (tid < p.Sk) kmv = p.keymask ? p.keymask[(size_t)b * p.Sk + tid] : 0.f;
    load_heads<KS_WARPS, 3>(dst, src, ld, rows, fill, tid);
    if (tid < AT_S) sm.kmask[tid] = kmv;
  }
  __syncthreads();
  const int k0 = warp * 16;   // this warp's keys
  float s[2][4];
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) s[nt][i] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a[4], bb[4];
    frag_a(a, sm.q, 0, kk * 16, lane);
    frag_b2(bb, sm.k, k0, kk * 16, lane);
    mma2(s[0], s[1], a, bb);
  }
  float mx[2] = {-INFINITY, -INFINITY};
#pragma unroll
  for (int nt = 0; nt < 2; ++nt) {
    const float2 ka = *reinterpret_cast<const float2*>(sm.kmask + k0 + nt * 8 + 2 * t);
    s[nt][0] += ka.x; s[nt][1] += ka.y; s[nt][2] += ka.x; s[nt][3] += ka.y;
#pragma unroll
    for (int i = 0; i < 4; ++i) mx[i >> 1] = fmaxf(mx[i >> 1], s[nt][i]);
  }
  float sum[2] = {0.f, 0.f};
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
    mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
  }
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      // a warp whose 16 keys all lie beyond Sk has m_w = -inf: its probabilities, sum and partial are exactly zero
      const float e = mx[i >> 1] == -INFINITY ? 0.f : __expf(s[nt][i] - mx[i >> 1]);
      s[nt][i] = e;
      sum[i >> 1] += e;
    }
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
    sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
  }
  if (t == 0) {
    sm.pm[warp][g] = mx[0]; sm.pm[warp][g + 8] = mx[1];
    sm.pl[warp][g] = sum[0]; sm.pl[warp][g + 8] = sum[1];
  }
  if (p.drop_thr) {
#pragma unroll
    for (int nt = 0; nt < 2; ++nt)
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        float d0, d1;
        vq_dropout_pair(p.seed, attn_pair_idx(vblk, g + r * 8, k0 + nt * 8 + 2 * t), p.drop_thr, p.drop_inv_keep, d0, d1);
        s[nt][2 * r] *= d0;
        s[nt][2 * r + 1] *= d1;
      }
  }
  // partial O_w = P_w V_w (un-normalised, relative to m_w)
  {
    uint32_t a[4];
    a[0] = pack_bf16(s[0][0], s[0][1]); a[1] = pack_bf16(s[0][2], s[0][3]);
    a[2] = pack_bf16(s[1][0], s[1][1]); a[3] = pack_bf16(s[1][2], s[1][3]);
    float o[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) o[nt][i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; nt += 2) {
      uint32_t bb[4];
      frag_b2_t(bb, sm.v, nt * 8, k0, lane);
      mma2(o[nt], o[nt + 1], a, bb);
    }
    __syncwarp();   // every lane has read its K / V fragments: the warp's rows of both tiles may now hold the partial
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = g + r * 8;
      if (qi < p.Sq) {
        float* dst = ks_partial_row(sm.k, sm.v, warp, qi) + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) *reinterpret_cast<float2*>(dst + nt * 8) = make_float2(o[nt][2 * r], o[nt][2 * r + 1]);
      }
    }
  }
  __syncthreads();
  // merge, normalise and write: thread -> (row = tid / 8, 8 columns)
  {
    const int qi = tid >> 3, c0 = (tid & 7) * 8;
    if (qi < p.Sq) {
      const float m = fmaxf(fmaxf(sm.pm[0][qi], sm.pm[1][qi]), fmaxf(sm.pm[2][qi], sm.pm[3][qi]));   // finite: key 0 always exists
      float l = 0.f, acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
      for (int w = 0; w < KS_WARPS; ++w) {
        const float sc = __expf(sm.pm[w][qi] - m);   // exp(-inf) = 0 for a warp without keys
        l += sc * sm.pl[w][qi];
        const float* so = ks_partial_row(sm.k, sm.v, w, qi) + c0;
        const float4 x = *reinterpret_cast<const float4*>(so), y = *reinterpret_cast<const float4*>(so + 4);
        acc[0] += sc * x.x; acc[1] += sc * x.y; acc[2] += sc * x.z; acc[3] += sc * x.w;
        acc[4] += sc * y.x; acc[5] += sc * y.y; acc[6] += sc * y.z; acc[7] += sc * y.w;
      }
      const float inv = 1.f / l;
      uint4 out;
      out.x = pack_bf16(acc[0] * inv, acc[1] * inv); out.y = pack_bf16(acc[2] * inv, acc[3] * inv);
      out.z = pack_bf16(acc[4] * inv, acc[5] * inv); out.w = pack_bf16(acc[6] * inv, acc[7] * inv);
      __nv_bfloat16* dst = p.o + (size_t)b * (p.o_bstride ? p.o_bstride : (long long)p.Sq * p.ldo) + (size_t)qi * p.ldo + h * AT_D + c0;
      *reinterpret_cast<uint4*>(dst) = out;
      if (c0 == 0 && p.lse) p.lse[((size_t)b * p.H + h) * p.Sq + qi] = m + __logf(l);
    }
  }
}

struct KsSmemBwd {
  __nv_bfloat16 q[16][AT_P], dO[16][AT_P], k[AT_S][AT_P], v[AT_S][AT_P];
  __nv_bfloat16 P[KS_WARPS][16][24], dS[KS_WARPS][16][24];   // per-warp [query][its 16 keys], 48-byte rows (ldmatrix-aligned)
  float kmask[AT_S];
  float D[16], lse[16];
  // followed by the per-warp fp32 dQ partials [KS_WARPS][Sq][KS_OP] (size depends on Sq, see ks_bwd_smem)
};
static inline int ks_bwd_smem(int Sq) { return (int)sizeof(KsSmemBwd) + KS_WARPS * Sq * KS_OP * 4; }

__global__ void __launch_bounds__(KS_WARPS * 32, 6) attn_ks_bwd_kernel(const AttnArgs p) {
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  KsSmemBwd& sm = *reinterpret_cast<KsSmemBwd*>(at_smem_base);
  float* dq_part = reinterpret_cast<float*>(at_smem_base + sizeof(KsSmemBwd));
  const int vblk = blockIdx.x, b = vblk / p.H, h = vblk % p.H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  {
    const AttnTile dst[4] = {sm.q, sm.dO, sm.k, sm.v};
    const __nv_bfloat16* const src[4] = {p.q + (size_t)b * p.Sq * p.ldq + h * AT_D, p.dO + (size_t)b * p.Sq * p.ldo + h * AT_D,
                                         p.k + (size_t)b * p.Sk * p.ldk + h * AT_D, p.v + (size_t)b * p.Sk * p.ldv + h * AT_D};
    const int ld[4] = {p.ldq, p.ldo, p.ldk, p.ldv};
    const int rows[4] = {p.Sq, p.Sq, p.Sk, p.Sk};
    const int fill[4] = {16, 16, AT_S, AT_S};
    float kmv = -INFINITY;
    if (tid < p.Sk) kmv = p.keymask ? p.keymask[(size_t)b * p.Sk + tid] : 0.f;
    // D[q] = sum_d dO[q][d] * O[q][d]: 8 threads per query row, 8 columns each. Its two loads are issued BEFORE the tile loads
    // and consumed after them: one DRAM round trip for everything instead of two in a row at the head of a 7 us CTA.
    const int qi = tid >> 3, c0 = (tid & 7) * 8;
    uint4 da = make_uint4(0, 0, 0, 0), oa = make_uint4(0, 0, 0, 0);
    float lse_q = INFINITY;                                                                    // rows >= Sq -> P = 0
    if (qi < p.Sq) {
      da = *reinterpret_cast<const uint4*>(p.dO + ((size_t)b * p.Sq + qi) * p.ldo + h * AT_D + c0);
      oa = *reinterpret_cast<const uint4*>(p.o_saved + ((size_t)b * p.Sq + qi) * p.ldo + h * AT_D + c0);
      if ((tid & 7) == 0) lse_q = p.lse[((size_t)b * p.H + h) * p.Sq + qi];
    }
    load_heads<KS_WARPS, 4>(dst, src, ld, rows, fill, tid);
    if (tid < AT_S) sm.kmask[tid] = kmv;
    {
      float acc = 0.f;
      const uint32_t aa[4] = {da.x, da.y, da.z, da.w}, oo[4] = {oa.x, oa.y, oa.z, oa.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 x = unpack_bf16(aa[j]), y = unpack_bf16(oo[j]);
        acc += x.x * y.x + x.y * y.y;
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if ((tid & 7) == 0) {
        sm.D[qi] = acc;
        sm.lse[qi] = lse_q;
      }
    }
  }
  __syncthreads();
  const int k0 = warp * 16;
  float s[2][4], dp[2][4];
#pragma unroll
  for (int nt = 0; nt < 2; ++nt)
#pragma unroll
    for (int i = 0; i < 4; ++i) s[nt][i] = dp[nt][i] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a[4], a2[4], bk[4], bv[4];
    frag_a(a, sm.q, 0, kk * 16, lane);
    frag_a(a2, sm.dO, 0, kk * 16, lane);
    frag_b2(bk, sm.k, k0, kk * 16, lane);
    frag_b2(bv, sm.v, k0, kk * 16, lane);
    mma2(s[0], s[1], a, bk);       // S = Q K_w^T
    mma2(dp[0], dp[1], a2, bv);    // dPd = dO V_w^T
  }
  const float lse[2] = {sm.lse[g], sm.lse[g + 8]};
  const float Dr[2] = {sm.D[g], sm.D[g + 8]};
#pragma unroll
  for (int nt = 0; nt < 2; ++nt) {
    const float2 ka = *reinterpret_cast<const float2*>(sm.kmask + k0 + nt * 8 + 2 * t);
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      float sc0 = 1.f, sc1 = 1.f;
      if (p.drop_thr) vq_dropout_pair(p.seed, attn_pair_idx(vblk, g + r * 8, k0 + nt * 8 + 2 * t), p.drop_thr, p.drop_inv_keep, sc0, sc1);
      const float p0 = __expf(s[nt][2 * r] + ka.x - lse[r]), p1 = __expf(s[nt][2 * r + 1] + ka.y - lse[r]);
      const float ds0 = p0 * (dp[nt][2 * r] * sc0 - Dr[r]), ds1 = p1 * (dp[nt][2 * r + 1] * sc1 - Dr[r]);
      s[nt][2 * r] = ds0; s[nt][2 * r + 1] = ds1;
      *reinterpret_cast<uint32_t*>(&sm.P[warp][g + r * 8][nt * 8 + 2 * t]) = pack_bf16(p0 * sc0, p1 * sc1);
      *reinterpret_cast<uint32_t*>(&sm.dS[warp][g + r * 8][nt * 8 + 2 * t]) = pack_bf16(ds0, ds1);
    }
  }
  // partial dQ = dS_w K_w, summed over warps with shared atomics
  {
    uint32_t a[4];
    a[0] = pack_bf16(s[0][0], s[0][1]); a[1] = pack_bf16(s[0][2], s[0][3]);
    a[2] = pack_bf16(s[1][0], s[1][1]); a[3] = pack_bf16(s[1][2], s[1][3]);
    float dq[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) dq[nt][i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; nt += 2) {
      uint32_t bb[4];
      frag_b2_t(bb, sm.k, nt * 8, k0, lane);
      mma2(dq[nt], dq[nt + 1], a, bb);
    }
    // parked per warp and summed after the barrier (fp32 shared atomicAdd would be a CAS loop per element)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = g + r * 8;
      if (qi < p.Sq) {
        float* dst = dq_part + ((size_t)warp * p.Sq + qi) * KS_OP + 2 * t;
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) *reinterpret_cast<float2*>(dst + nt * 8) = make_float2(dq[nt][2 * r], dq[nt][2 * r + 1]);
      }
    }
  }
  __syncwarp();
  // dV_w = Pd_w^T dO, dK_w = dS_w^T Q  (A = transposed per-warp tile [16 keys x 16 queries]; one k-step over the 16 query slots)
  if (k0 < p.Sk) {
    uint32_t ap[4], as[4];
    {
      const int mi = lane >> 3, r = lane & 7;
      ldsm_x4_t(ap, &sm.P[warp][(mi >> 1) * 8 + r][(mi & 1) * 8]);
      ldsm_x4_t(as, &sm.dS[warp][(mi >> 1) * 8 + r][(mi & 1) * 8]);
    }
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[nt][i] = dk[nt][i] = 0.f;
#pragma unroll
    for (int nt = 0; nt < 8; nt += 2) {
      uint32_t b1[4], b2[4];
      frag_b2_t(b1, sm.dO, nt * 8, 0, lane);
      frag_b2_t(b2, sm.q, nt * 8, 0, lane);
      mma2(dv[nt], dv[nt + 1], ap, b1);
      mma2(dk[nt], dk[nt + 1], as, b2);
    }
    // rows [k0, k0 + 16) of the k / v tiles are only ever read by this warp, and it is done with them: stage dK / dV there
    store_tile16(sm.k, k0, dk, p.dk + (size_t)b * p.Sk * p.lddk + h * AT_D, p.lddk, p.Sk, lane);
    store_tile16(sm.v, k0, dv, p.dv + (size_t)b * p.Sk * p.lddv + h * AT_D, p.lddv, p.Sk, lane);
  }
  __syncthreads();
  {
    const int qi = tid >> 3, c0 = (tid & 7) * 8;
    if (qi < p.Sq) {
      float acc[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = 0.f;
#pragma unroll
      for (int w = 0; w < KS_WARPS; ++w) {
        const float* so = dq_part + ((size_t)w * p.Sq + qi) * KS_OP + c0;
        const float4 x = *reinterpret_cast<const float4*>(so), y = *reinterpret_cast<const float4*>(so + 4);
        acc[0] += x.x; acc[1] += x.y; acc[2] += x.z; acc[3] += x.w; acc[4] += y.x; acc[5] += y.y; acc[6] += y.z; acc[7] += y.w;
      }
      uint4 out;
      out.x = pack_bf16(acc[0], acc[1]); out.y = pack_bf16(acc[2], acc[3]); out.z = pack_bf16(acc[4], acc[5]); out.w = pack_bf16(acc[6], acc[7]);
      *reinterpret_cast<uint4*>(p.dq + ((size_t)b * p.Sq + qi) * p.lddq + h * AT_D + c0) = out;
    }
  }
}


// =====================================================================================================================
// Generic multi-tile kernels: up to MT_MAX queries x MT_MAX keys per (batch, head) problem, in 64 x 64 tiles. They serve the
// shapes the single-tile kernels above reject — a longer visual sequence (BASELINE.json configs[3]: NExT-QA-style clip
// features, L + N up to 254 encoder tokens, and the decoder's cross-attention to those L + N + 2 memory rows). One 4-warp
// CTA owns one problem and keeps Q, K, V (backward: + dO) of the whole problem in shared memory.
//   forward : per 64-row query tile, flash-style online softmax over the key tiles (running max / sum / O in registers)
//   backward: P is recomputed from the saved log-sum-exp, D = rowsum(dO * O) from the saved output.
//             pass A — query tile outer, key tile inner: dQ accumulates in registers;
//             pass B — key tile outer, query tile inner: P / dS of the tile pair go through two shared 64 x 64 tiles and
//             dK / dV accumulate in registers (the tile math is done twice; QK^T / PV are ~1 % of the step's FLOPs).
// The relative-position bias exists only between text tokens (Lt <= 64), i.e. inside tile pair (0, 0).
// =====================================================================================================================
constexpr int MT_MAX = 256;
VQ_DEVINL uint32_t mt_pair_idx(uint32_t blk, int q, int k) { return ((blk * MT_MAX + (uint32_t)q) * MT_MAX + (uint32_t)k) >> 1; }
VQ_DEVINL int rows64(int n) { return (n + 63) & ~63; }
constexpr int MT_HDR_FLOATS = 2 * AT_S + MT_MAX + 64;   // bias[128] | kmask[256] | dbucket[64]
static inline int mt_smem_fwd(int Sq, int Sk) { return MT_HDR_FLOATS * 4 + (((Sq + 15) & ~15) + 2 * ((Sk + 63) & ~63)) * AT_P * 2; }
static inline int mt_smem_bwd(int Sq, int Sk) {
  return MT_HDR_FLOATS * 4 + 2 * MT_MAX * 4 + (2 * ((Sq + 15) & ~15) + 2 * ((Sk + 63) & ~63) + 2 * AT_S) * AT_P * 2;
}

template <int NW>
VQ_DEVINL void mt_load_header(float* sbias, float* skmask, const AttnArgs& p, const AttnBuckets& bk, int b, int h, int tid) {
  if (p.rel_mode)
    for (int r = tid; r < 2 * AT_S - 1; r += NW * 32) sbias[r] = p.rel_table[(int)bk.b[r] * p.H + h];
  for (int j = tid; j < MT_MAX; j += NW * 32) skmask[j] = j < p.Sk ? (p.keymask ? p.keymask[(size_t)b * p.Sk + j] : 0.f) : -INFINITY;
}

__global__ void __launch_bounds__(128) attn_mt_fwd_kernel(const AttnArgs p, const __grid_constant__ AttnBuckets bk) {
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  const int vblk = blockIdx.x, b = vblk / p.H, h = vblk % p.H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  float* sbias = reinterpret_cast<float*>(at_smem_base);
  float* skmask = sbias + 2 * AT_S;
  AttnTile sq = reinterpret_cast<AttnTile>(at_smem_base + MT_HDR_FLOATS * 4);
  AttnTile sk = sq + rows16(p.Sq);
  AttnTile sv = sk + rows64(p.Sk);
  {
    const AttnTile dst[3] = {sq, sk, sv};
    const __nv_bfloat16* const src[3] = {p.q + (size_t)b * (p.q_bstride ? p.q_bstride : (long long)p.Sq * p.ldq) + h * AT_D,
                                         p.k + (size_t)b * (p.k_bstride ? p.k_bstride : (long long)p.Sk * p.ldk) + h * AT_D,
                                         p.v + (size_t)b * (p.v_bstride ? p.v_bstride : (long long)p.Sk * p.ldv) + h * AT_D};
    const int ld[3] = {p.ldq, p.ldk, p.ldv};
    const int rows[3] = {p.Sq, p.Sk, p.Sk};
    const int fill[3] = {rows16(p.Sq), rows64(p.Sk), rows64(p.Sk)};
    mt_load_header<4>(sbias, skmask, p, bk, b, h, tid);
    load_heads<4, 3>(dst, src, ld, rows, fill, tid);
  }
  __syncthreads();
  const int nqt = (p.Sq + 63) >> 6, nkt = (p.Sk + 63) >> 6;
  for (int i = 0; i < nqt; ++i) {
    const int m0 = warp * 16, qrow0 = i * 64 + m0;
    if (qrow0 >= p.Sq) continue;                           // no barrier inside this loop: warps are independent
    float mrun[2] = {-INFINITY, -INFINITY}, lrun[2] = {0.f, 0.f};
    float o[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int x = 0; x < 4; ++x) o[nt][x] = 0.f;
    for (int j = 0; j < nkt; ++j) {
      AttnArgs pt = p;
      pt.rel_mode = (i == 0 && j == 0) ? p.rel_mode : 0;   // bias only in the text x text corner
      pt.causal = 0;
      float s[8][4];
      scores_tile<8>(s, sq + i * 64, sk + j * 64, sbias, skmask + j * 64, pt, m0, lane);
      float mx[2] = {mrun[0], mrun[1]};
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int x = 0; x < 4; ++x) mx[x >> 1] = fmaxf(mx[x >> 1], s[nt][x]);
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 1));
        mx[r] = fmaxf(mx[r], __shfl_xor_sync(0xffffffffu, mx[r], 2));
      }
      float sc[2], sum[2] = {0.f, 0.f};
#pragma unroll
      for (int r = 0; r < 2; ++r) sc[r] = mrun[r] == -INFINITY ? 0.f : __expf(mrun[r] - mx[r]);   // key 0 exists: mx is finite
#pragma unroll
      for (int nt = 0; nt < 8; ++nt)
#pragma unroll
        for (int x = 0; x < 4; ++x) {
          const float e = __expf(s[nt][x] - mx[x >> 1]);
          s[nt][x] = e;
          sum[x >> 1] += e;
        }
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 1);
        sum[r] += __shfl_xor_sync(0xffffffffu, sum[r], 2);
        lrun[r] = lrun[r] * sc[r] + sum[r];
        mrun[r] = mx[r];
      }
#pragma unroll
      for (int nt = 0; nt < 8; ++nt) {
        o[nt][0] *= sc[0]; o[nt][1] *= sc[0]; o[nt][2] *= sc[1]; o[nt][3] *= sc[1];
      }
      if (p.drop_thr) {
#pragma unroll
        for (int nt = 0; nt < 8; ++nt)
#pragma unroll
          for (int r = 0; r < 2; ++r) {
            float d0, d1;
            vq_dropout_pair(p.seed, mt_pair_idx(vblk, qrow0 + g + r * 8, j * 64 + nt * 8 + 2 * t), p.drop_thr, p.drop_inv_keep, d0, d1);
            s[nt][2 * r] *= d0;
            s[nt][2 * r + 1] *= d1;
          }
      }
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        uint32_t a[4];
        a[0] = pack_bf16(s[2 * kk][0], s[2 * kk][1]);
        a[1] = pack_bf16(s[2 * kk][2], s[2 * kk][3]);
        a[2] = pack_bf16(s[2 * kk + 1][0], s[2 * kk + 1][1]);
        a[3] = pack_bf16(s[2 * kk + 1][2], s[2 * kk + 1][3]);
#pragma unroll
        for (int nt = 0; nt < 8; nt += 2) {
          uint32_t bb[4];
          frag_b2_t(bb, sv + j * 64, nt * 8, kk * 16, lane);
          mma2(o[nt], o[nt + 1], a, bb);
        }
      }
    }
    const float inv[2] = {1.f / lrun[0], 1.f / lrun[1]};
#pragma unroll
    for (int nt = 0; nt < 8; ++nt) {
      o[nt][0] *= inv[0]; o[nt][1] *= inv[0]; o[nt][2] *= inv[1]; o[nt][3] *= inv[1];
    }
    if (t == 0 && p.lse) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int qi = qrow0 + g + r * 8;
        if (qi < p.Sq) p.lse[((size_t)b * p.H + h) * p.Sq + qi] = mrun[r] + __logf(lrun[r]);
      }
    }
    // this warp's 16 rows of the q tile are dead: stage O there and write full 128-byte rows
    store_tile16(sq + i * 64, m0, o, p.o + (size_t)b * (p.o_bstride ? p.o_bstride : (long long)p.Sq * p.ldo) + (size_t)i * 64 * p.ldo + h * AT_D,
                 p.ldo, p.Sq - i * 64, lane);
  }
}

struct MtSmemB { float *bias, *kmask, *dbucket, *lse, *D; AttnTile q, dO, k, v, P, dS; };

// P and dS of the tile pair (query tile i rows [16 warp, 16 warp + 16), key tile j) in the m16n8 accumulator layout of this
// warp: ds[nt][x]; optionally also written (P with the dropout scale folded in, for dV) to the shared P / dS tiles
template <bool STORE>
VQ_DEVINL void mt_tile_p_ds(float (&ds)[8][4], const AttnArgs& p, const MtSmemB& sm, int vblk, int i, int j, int m0, int lane) {
  const int g = lane >> 2, t = lane & 3;
  AttnArgs pt = p;
  pt.rel_mode = (i == 0 && j == 0) ? p.rel_mode : 0;
  pt.causal = 0;
  float s[8][4], dp[8][4];
  scores_tile<8>(s, sm.q + i * 64, sm.k + j * 64, sm.bias, sm.kmask + j * 64, pt, m0, lane);
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int x = 0; x < 4; ++x) dp[nt][x] = 0.f;
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) {
    uint32_t a[4];
    frag_a(a, sm.dO + i * 64, m0, kk * 16, lane);
#pragma unroll
    for (int nt = 0; nt < 8; nt += 2) {
      uint32_t bb[4];
      frag_b2(bb, sm.v + j * 64, nt * 8, kk * 16, lane);
      mma2(dp[nt], dp[nt + 1], a, bb);
    }
  }
  float lse[2], Dr[2];
#pragma unroll
  for (int r = 0; r < 2; ++r) {
    const int qi = i * 64 + m0 + g + r * 8;
    lse[r] = qi < p.Sq ? sm.lse[qi] : INFINITY;     // rows >= Sq: P = 0
    Dr[r] = qi < p.Sq ? sm.D[qi] : 0.f;
  }
#pragma unroll
  for (int nt = 0; nt < 8; ++nt)
#pragma unroll
    for (int r = 0; r < 2; ++r) {
      const int qi = i * 64 + m0 + g + r * 8, kj = j * 64 + nt * 8 + 2 * t;
      float sc0 = 1.f, sc1 = 1.f;
      if (p.drop_thr) vq_dropout_pair(p.seed, mt_pair_idx(vblk, qi, kj), p.drop_thr, p.drop_inv_keep, sc0, sc1);
      const float p0 = __expf(s[nt][2 * r] - lse[r]), p1 = __expf(s[nt][2 * r + 1] - lse[r]);
      const float d0 = p0 * (dp[nt][2 * r] * sc0 - Dr[r]), d1 = p1 * (dp[nt][2 * r + 1] * sc1 - Dr[r]);
      ds[nt][2 * r] = d0;
      ds[nt][2 * r + 1] = d1;
      if (STORE) {
        *reinterpret_cast<uint32_t*>(&sm.P[m0 + g + r * 8][nt * 8 + 2 * t]) = pack_bf16(p0 * sc0, p1 * sc1);
        *reinterpret_cast<uint32_t*>(&sm.dS[m0 + g + r * 8][nt * 8 + 2 * t]) = pack_bf16(d0, d1);
      }
    }
}

__global__ void __launch_bounds__(128) attn_mt_bwd_kernel(const AttnArgs p, const __grid_constant__ AttnBuckets bk) {
  vq_pdl_trigger();
  vq_pdl_wait();
  extern __shared__ __align__(16) uint8_t at_smem_base[];
  const int vblk = blockIdx.x, b = vblk / p.H, h = vblk % p.H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  MtSmemB sm;
  sm.bias = reinterpret_cast<float*>(at_smem_base);
  sm.kmask = sm.bias + 2 * AT_S;
  sm.dbucket = sm.kmask + MT_MAX;
  sm.lse = sm.dbucket + 64;
  sm.D = sm.lse + MT_MAX;
  sm.q = reinterpret_cast<AttnTile>(at_smem_base + (MT_HDR_FLOATS + 2 * MT_MAX) * 4);
  sm.dO = sm.q + rows16(p.Sq);
  sm.k = sm.dO + rows16(p.Sq);
  sm.v = sm.k + rows64(p.Sk);
  sm.P = sm.v + rows64(p.Sk);
  sm.dS = sm.P + AT_S;
  {
    const AttnTile dst[4] = {sm.q, sm.dO, sm.k, sm.v};
    const __nv_bfloat16* const src[4] = {p.q + (size_t)b * p.Sq * p.ldq + h * AT_D, p.dO + (size_t)b * p.Sq * p.ldo + h * AT_D,
                                         p.k + (size_t)b * p.Sk * p.ldk + h * AT_D, p.v + (size_t)b * p.Sk * p.ldv + h * AT_D};
    const int ld[4] = {p.ldq, p.ldo, p.ldk, p.ldv};
    const int rows[4] = {p.Sq, p.Sq, p.Sk, p.Sk};
    const int fill[4] = {rows16(p.Sq), rows16(p.Sq), rows64(p.Sk), rows64(p.Sk)};
    mt_load_header<4>(sm.bias, sm.kmask, p, bk, b, h, tid);
    for (int x = tid; x < 64; x += 128) sm.dbucket[x] = 0.f;
    // D[q] = sum_d dO[q][d] * O[q][d] (the saved forward output), lse[q]: 8 threads per row
    for (int base = 0; base < p.Sq; base += 16) {
      const int qi = base + (tid >> 3), c0 = (tid & 7) * 8;
      float acc = 0.f;
      if (qi < p.Sq) {
        const uint4 a = *reinterpret_cast<const uint4*>(p.dO + ((size_t)b * p.Sq + qi) * p.ldo + h * AT_D + c0);
        const uint4 o = *reinterpret_cast<const uint4*>(p.o_saved + ((size_t)b * p.Sq + qi) * p.ldo + h * AT_D + c0);
        const uint32_t aa[4] = {a.x, a.y, a.z, a.w}, oo[4] = {o.x, o.y, o.z, o.w};
#pragma unroll
        for (int x = 0; x < 4; ++x) {
          const float2 u = unpack_bf16(aa[x]), w = unpack_bf16(oo[x]);
          acc += u.x * w.x + u.y * w.y;
        }
      }
      acc += __shfl_xor_sync(0xffffffffu, acc, 1);
      acc += __shfl_xor_sync(0xffffffffu, acc, 2);
      acc += __shfl_xor_sync(0xffffffffu, acc, 4);
      if ((tid & 7) == 0 && qi < p.Sq) {
        sm.D[qi] = acc;
        sm.lse[qi] = p.lse[((size_t)b * p.H + h) * p.Sq + qi];
      }
    }
    load_heads<4, 4>(dst, src, ld, rows, fill, tid);
  }
  __syncthreads();
  const int nqt = (p.Sq + 63) >> 6, nkt = (p.Sk + 63) >> 6;
  const int m0 = warp * 16;
  // ---- pass A: dQ (and the bias-table gradient from tile pair (0, 0)) ----
  for (int i = 0; i < nqt; ++i) {
    const bool has_q = i * 64 + m0 < p.Sq;
    float dq[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int x = 0; x < 4; ++x) dq[nt][x] = 0.f;
    for (int j = 0; j < nkt; ++j) {
      const bool bias_tile = p.d_rel_table && p.rel_mode && i == 0 && j == 0;
      float ds[8][4];
      if (has_q) {
        if (bias_tile) mt_tile_p_ds<true>(ds, p, sm, vblk, i, j, m0, lane);
        else mt_tile_p_ds<false>(ds, p, sm, vblk, i, j, m0, lane);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          uint32_t a[4];
          a[0] = pack_bf16(ds[2 * kk][0], ds[2 * kk][1]);
          a[1] = pack_bf16(ds[2 * kk][2], ds[2 * kk][3]);
          a[2] = pack_bf16(ds[2 * kk + 1][0], ds[2 * kk + 1][1]);
          a[3] = pack_bf16(ds[2 * kk + 1][2], ds[2 * kk + 1][3]);
#pragma unroll
          for (int nt = 0; nt < 8; nt += 2) {
            uint32_t bb[4];
            frag_b2_t(bb, sm.k + j * 64, nt * 8, kk * 16, lane);
            mma2(dq[nt], dq[nt + 1], a, bb);
          }
        }
      }
      if (bias_tile) {      // block-uniform condition
        __syncthreads();
        const int nq = min(p.Sq, p.Lt), nk = min(p.Sk, p.Lt);
        const int ndiag = nq + nk - 1;
        for (int dgi = tid; dgi < ndiag; dgi += 128) {
          const int rel = dgi - (nq - 1);
          const int q_lo = max(0, -rel), q_hi = min(nq, nk - rel);
          float acc = 0.f;
          for (int qi = q_lo; qi < q_hi; ++qi) acc += __bfloat162float(sm.dS[qi][qi + rel]);
          if (q_hi > q_lo) atomicAdd(&sm.dbucket[(int)bk.b[rel + (AT_S - 1)]], acc);
        }
        __syncthreads();
        for (int x = tid; x < 64; x += 128) {
          const float v = sm.dbucket[x];
          if (v != 0.f) atomicAdd(&p.d_rel_table[x * p.H + h], v);
        }
      }
    }
    if (has_q) {
#pragma unroll
      for (int r = 0; r < 2; ++r) {
        const int qi = i * 64 + m0 + g + r * 8;
        if (qi < p.Sq) {
          __nv_bfloat16* dst = p.dq + ((size_t)b * p.Sq + qi) * p.lddq + h * AT_D + 2 * t;
#pragma unroll
          for (int nt = 0; nt < 8; ++nt) *reinterpret_cast<uint32_t*>(dst + nt * 8) = pack_bf16(dq[nt][2 * r], dq[nt][2 * r + 1]);
        }
      }
    }
  }
  // ---- pass B: dK, dV ----
  for (int j = 0; j < nkt; ++j) {
    const bool has_k = j * 64 + m0 < p.Sk;
    float dv[8][4], dk[8][4];
#pragma unroll
    for (int nt = 0; nt < 8; ++nt)
#pragma unroll
      for (int x = 0; x < 4; ++x) dv[nt][x] = dk[nt][x] = 0.f;
    for (int i = 0; i < nqt; ++i) {
      __syncthreads();                                   // the previous tile pair's P / dS have been consumed
      if (i * 64 + m0 < p.Sq) {
        float ds[8][4];
        mt_tile_p_ds<true>(ds, p, sm, vblk, i, j, m0, lane);
      } else {
        // this warp has no query rows in tile i: its 16 rows of P / dS must read as zero in the contraction below
        for (int x = lane; x < 16 * (AT_D / 8); x += 32) {
          *reinterpret_cast<uint4*>(&sm.P[m0 + (x >> 3)][(x & 7) * 8]) = make_uint4(0, 0, 0, 0);
          *reinterpret_cast<uint4*>(&sm.dS[m0 + (x >> 3)][(x & 7) * 8]) = make_uint4(0, 0, 0, 0);
        }
      }
      __syncthreads();
      if (has_k) {
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
          if (i * 64 + kk * 16 < p.Sq) {
            uint32_t ap[4], as[4];
            frag_a_t(ap, sm.P, m0, kk * 16, lane);
            frag_a_t(as, sm.dS, m0, kk * 16, lane);
#pragma unroll
            for (int nt = 0; nt < 8; nt += 2) {
              uint32_t b1[4], b2[4];
              frag_b2_t(b1, sm.dO + i * 64, nt * 8, kk * 16, lane);
              frag_b2_t(b2, sm.q + i * 64, nt * 8, kk * 16, lane);
              mma2(dv[nt], dv[nt + 1], ap, b1);
              mma2(dk[nt], dk[nt + 1], as, b2);
            }
          }
        }
      }
    }
    __syncthreads();      // every warp is done reading K_j / V_j (scores, dP) before their rows become staging space
    if (has_k) {
      store_tile16(sm.k + j * 64, m0, dk, p.dk + ((size_t)b * p.Sk + (size_t)j * 64) * p.lddk + h * AT_D, p.lddk, p.Sk - j * 64, lane);
      store_tile16(sm.v + j * 64, m0, dv, p.dv + ((size_t)b * p.Sk + (size_t)j * 64) * p.lddv + h * AT_D, p.lddv, p.Sk - j * 64, lane);
    }
  }
}

static int launch_mt_fwd(const AttnArgs& a, const AttnBuckets& bk, cudaStream_t stream) {
  const int smem = mt_smem_fwd(a.Sq, a.Sk);
  static int attr_smem = 0;
  if (smem > attr_smem) {
    VQ_CUDA(cudaFuncSetAttribute(attn_mt_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, mt_smem_fwd(MT_MAX, MT_MAX)));
    attr_smem = mt_smem_fwd(MT_MAX, MT_MAX);
  }
  (void)vq_launch(attn_mt_fwd_kernel, dim3(a.B * a.H), dim3(128), (size_t)smem, stream, a, bk);
  VQ_LAUNCH_CHECK();
  return 0;
}
static int launch_mt_bwd(const AttnArgs& a, const AttnBuckets& bk, cudaStream_t stream) {
  VQ_CHECK(a.o_saved, "attention bwd: the multi-tile backward needs the saved forward output (o_saved)");
  const int smem = mt_smem_bwd(a.Sq, a.Sk);
  static int attr_smem = 0;
  if (smem > attr_smem) {
    VQ_CUDA(cudaFuncSetAttribute(attn_mt_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, mt_smem_bwd(MT_MAX, MT_MAX)));
    attr_smem = mt_smem_bwd(MT_MAX, MT_MAX);
  }
  (void)vq_launch(attn_mt_bwd_kernel, dim3(a.B * a.H), dim3(128), (size_t)smem, stream, a, bk);
  VQ_LAUNCH_CHECK();
  return 0;
}

static int check_args(const AttnArgs& a) {
  VQ_CHECK(a.Sq >= 1 && a.Sq <= MT_MAX && a.Sk >= 1 && a.Sk <= MT_MAX, "attention: Sq=%d Sk=%d must be in [1,%d]", a.Sq, a.Sk, MT_MAX);
  if (a.Sq > AT_S || a.Sk > AT_S) {
    VQ_CHECK(!a.causal && a.rel_mode != 2, "attention: causal / everywhere-biased (decoder self-) attention is limited to %d positions", AT_S);
    VQ_CHECK(a.rel_mode == 0 || a.Lt <= AT_S, "attention: the biased text x text corner must fit one tile (Lt=%d)", a.Lt);
    VQ_CHECK(!a.q_off, "attention: multi-tile problems take no query offset");
  }
  VQ_CHECK(a.q_off == 0 || (a.q_off > 0 && a.q_off + a.Sq <= AT_S),
           "attention: q_off=%d with Sq=%d leaves the %d positions of the relative-position window", a.q_off, a.Sq, AT_S);
  VQ_CHECK(a.ldq % 8 == 0 && a.ldk % 8 == 0 && a.ldv % 8 == 0 && a.ldo % 8 == 0, "attention: pitches must be multiples of 8");
  VQ_CHECK(a.rel_mode == 0 || (a.rel_table && a.rel_bucket), "attention: rel_mode needs rel_table and rel_bucket");
  return 0;
}

static int make_buckets(const AttnArgs& a, AttnBuckets* bk) {
  memset(bk, 0, sizeof(*bk));
  if (a.rel_mode)
    for (int r = 0; r < 2 * AT_S - 1; ++r) {
      VQ_CHECK(a.rel_bucket[r] >= 0 && a.rel_bucket[r] < 64, "attention: bucket %d out of range", a.rel_bucket[r]);
      bk->b[r] = (int8_t)a.rel_bucket[r];
    }
  return 0;
}

constexpr int AT_HPC = 4;   // single-warp problems per CTA
template <int NW, int NKT>
static int launch_fwd(const AttnArgs& a, const AttnBuckets& bk, cudaStream_t stream) {
  constexpr int HPC = NW == 1 ? AT_HPC : 1;
  constexpr int STAGES = NW == 4 ? 2 : 1;       // NW == 4: persistent CTAs with two cp.async stages, 3 CTAs per SM
  static bool attr = false;
  if (!attr) {
    VQ_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<NW, NKT, HPC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 STAGES * HPC * attn_smem_fwd(NW * 16, NKT * 8)));
    VQ_CUDA(cudaFuncSetAttribute(attn_fwd_kernel<NW, NKT, HPC>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr = true;
  }
  int grid = (a.B * a.H + HPC - 1) / HPC;
  if (NW == 4 && grid > 3 * num_sms()) grid = 3 * num_sms();
  (void)vq_launch(attn_fwd_kernel<NW, NKT, HPC>, dim3(grid), dim3(32 * NW * HPC),
                  (size_t)STAGES * HPC * attn_smem_fwd(a.Sq, NKT * 8), stream, a, bk);
  VQ_LAUNCH_CHECK();
  return 0;
}
template <int NW, int NKT>
static int launch_bwd(const AttnArgs& a, const AttnBuckets& bk, cudaStream_t stream) {
  constexpr int HPC = NW == 1 ? AT_HPC : 1;
  static bool attr = false;
  if (!attr) {
    VQ_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<NW, NKT, HPC>, cudaFuncAttributeMaxDynamicSharedMemorySize, HPC * attn_smem_bwd(AT_S, NKT * 8)));
    VQ_CUDA(cudaFuncSetAttribute(attn_bwd_kernel<NW, NKT, HPC>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    attr = true;
  }
  (void)vq_launch(attn_bwd_kernel<NW, NKT, HPC>, dim3((a.B * a.H + HPC - 1) / HPC), dim3(32 * NW * HPC),
                  (size_t)HPC * attn_smem_bwd(a.Sq, NKT * 8), stream, a, bk);
  VQ_LAUNCH_CHECK();
  return 0;
}

int attn_fwd(const AttnArgs& a, cudaStream_t stream) {
  if (check_args(a)) return 1;
  AttnBuckets bk;
  if (make_buckets(a, &bk)) return 1;
  if (a.Sq > AT_S || a.Sk > AT_S) return launch_mt_fwd(a, bk, stream);   // longer visual sequence: generic multi-tile kernel
  if (attn_tc_eligible(a)) return attn_enc_fwd_tc(a, bk, stream);         // encoder: tcgen05 + TMA kernel (attention_tc.cu)
  const int warps = (a.Sq + 15) / 16;   // one warp per 16 query rows
  if (a.Sq <= 16 && a.Sk > 16 && a.rel_mode == 0 && !a.causal) {   // few queries, many keys (cross-attention): key-split kernel
    static bool attr = false;
    if (!attr) {
      VQ_CUDA(cudaFuncSetAttribute(attn_ks_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(KsSmemFwd)));
      attr = true;
    }
    (void)vq_launch(attn_ks_fwd_kernel, dim3(a.B * a.H), dim3(KS_WARPS * 32), sizeof(KsSmemFwd), stream, a);
    VQ_LAUNCH_CHECK();
    return 0;
  }
  if (warps == 1 && a.Sk <= 16) return launch_fwd<1, 2>(a, bk, stream);   // decoder self-attention / decode steps
  if (warps == 1) return launch_fwd<1, 8>(a, bk, stream);                  // cross-attention
  if (warps == 2) return launch_fwd<2, 8>(a, bk, stream);
  return launch_fwd<4, 8>(a, bk, stream);                                  // encoder
}

int attn_bwd(const AttnArgs& a, cudaStream_t stream) {
  if (check_args(a)) return 1;
  VQ_CHECK(a.lse && a.dO && a.dq && a.dk && a.dv, "attention bwd: missing pointers");
  VQ_CHECK(!a.q_bstride && !a.k_bstride && !a.v_bstride && !a.o_bstride && !a.q_off, "attention bwd: strided / offset form is forward-only");
  VQ_CHECK(a.lddq % 8 == 0 && a.lddk % 8 == 0 && a.lddv % 8 == 0, "attention bwd: pitches must be multiples of 8");
  AttnBuckets bk;
  if (make_buckets(a, &bk)) return 1;
  if (a.Sq > AT_S || a.Sk > AT_S) return launch_mt_bwd(a, bk, stream);
  if (attn_tc_bwd_eligible(a)) return attn_enc_bwd_tc(a, bk, stream);
  if (a.o_saved && a.Sq <= 16 && a.Sk > 16 && a.rel_mode == 0 && !a.causal) {   // key-split backward (needs the forward output)
    static bool attr = false;
    if (!attr) {
      VQ_CUDA(cudaFuncSetAttribute(attn_ks_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ks_bwd_smem(16)));
      attr = true;
    }
    (void)vq_launch(attn_ks_bwd_kernel, dim3(a.B * a.H), dim3(KS_WARPS * 32), (size_t)ks_bwd_smem(a.Sq), stream, a);
    VQ_LAUNCH_CHECK();
    return 0;
  }
  const int warps = (max(a.Sq, a.Sk) + 15) / 16;   // phase 1: 16 query rows per warp, phase 2: 16 key rows per warp
  if (warps == 1) return launch_bwd<1, 2>(a, bk, stream);
  if (warps == 2) return launch_bwd<2, 8>(a, bk, stream);
  return launch_bwd<4, 8>(a, bk, stream);
}

}  // namespace vq
