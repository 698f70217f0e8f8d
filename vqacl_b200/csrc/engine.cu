// VL-T5 / VQACL train step on B200: forward (VLT5.forward with labels, modeling_t5_our.py:514-713), backward and the
// clip + AdamW tail (vqacl.py:461-487), issued kernel by kernel from C++.
//
// Data layout in HBM
//   parameter arena  : one flat fp32 buffer (master weights), a same-shaped fp32 gradient arena and a bf16 copy that feeds
//                      the tensor cores. Fused weights are adjacent so one GEMM covers them: per layer [Wq;Wk;Wv] (N = 2304),
//                      and the cross-attention [Wk;Wv] of ALL decoder layers ([18432, 768]) so that the K/V projection of the
//                      [B,58,768] decoder memory is a single GEMM (62 % of the decoder's FLOPs, SURVEY.md §8a8).
//                      Order: decoder | cross-KV | encoder | visual | shared | no-decay group | never-trained group, i.e.
//                      the order in which backward finishes gradients (bucketed all-reduce) and the AdamW decay boundary.
//   residual stream  : fp32 snapshots x_k (one per sub-layer) so RMSNorm backward re-reads its exact input.
//   GEMM operands    : bf16, row-major [rows, features]; attention reads heads in place from the packed [rows, 2304] QKV.
#include "engine.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>

namespace vq {

// dropout site ids (the keep-mask of element i at site s is hash(seed, s, i); recomputed in backward, never stored)
enum : uint32_t { SITE_ENC_EMB = 1, SITE_ENC_FINAL = 2, SITE_DEC_EMB = 3, SITE_DEC_FINAL = 4 };
static inline uint32_t site_enc(int l, int k) { return 100u + (uint32_t)l * 4u + (uint32_t)k; }   // 0 probs 1 attn-out 2 ffn-inner 3 ffn-out
static inline uint32_t site_dec(int l, int k) { return 300u + (uint32_t)l * 8u + (uint32_t)k; }   // 0 self probs 1 self out 2 cross probs 3 cross out 4 ffn inner 5 ffn out

Dropout Engine::drop(uint32_t site) const {
  Dropout d;
  if (training && cfg.dropout > 0.f) {
    double t = floor((double)cfg.dropout * 65536.0 + 0.5);
    if (t < 1.0) t = 1.0;
    if (t > 65535.0) t = 65535.0;
    d.thr = (uint32_t)t;                                   // 16-bit threshold: p is quantised to 1/65536
    d.inv_keep = (float)(65536.0 / (65536.0 - t));
    uint64_t k = ((uint64_t)seed << 32 | site) * 0x9E3779B97F4A7C15ull;   // key = mix(seed, site), once per launch
    k ^= k >> 29; k *= 0xBF58476D1CE4E5B9ull; k ^= k >> 32;
    d.seed = (uint32_t)k;
    d.site = site;
  }
  return d;
}

// --------------------------------------------------------------------------------------------------- layout
static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int engine_build_layout(Engine& e) {
  const vqacl_config& c = e.cfg;
  VQ_CHECK(c.d_model == DM, "engine: kernels are specialised for d_model = %d (got %d)", DM, c.d_model);
  VQ_CHECK(c.d_kv == 64 && c.n_heads * c.d_kv == c.d_model, "engine: needs d_kv = 64 and n_heads * d_kv = d_model");
  VQ_CHECK(c.n_buckets <= 64, "engine: at most 64 relative-position buckets");
  VQ_CHECK(c.vocab_size % 8 == 0 && c.d_ff % 8 == 0 && c.feat_dim % 8 == 0, "engine: vocab, d_ff, feat_dim must be multiples of 8");
  const int d = c.d_model, f = c.d_ff;
  size_t off = 0;
  auto add = [&](const std::string& name, int rows, int cols, int group) {
    off = align_up(off, 64);
    e.params.push_back({name, off, rows, cols, group});
    const size_t o = off;
    off += (size_t)rows * cols;
    return o;
  };
  e.dec.resize(c.n_dec_layers);
  e.enc.resize(c.n_enc_layers);
  char b[256];
  // ---- weight-decay group -------------------------------------------------------------------------------
  // (1) the GEMM-only matrices, in the order backward finishes their gradients: with N > 1 GPUs this region is reduce-
  //     scattered bucket by bucket, every rank runs AdamW on its slices only and the refreshed bf16 copies are all-gathered
  for (int l = 0; l < c.n_dec_layers; ++l) {
    DecLayer& L = e.dec[l];
    snprintf(b, sizeof b, "decoder.block.%d.layer.0.SelfAttention.q.weight", l); L.qkv = add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.0.SelfAttention.k.weight", l); add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.0.SelfAttention.v.weight", l); add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.0.SelfAttention.o.weight", l); L.o = add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.1.EncDecAttention.q.weight", l); L.cq = add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.1.EncDecAttention.o.weight", l); L.co = add(b, d, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.2.DenseReluDense.wi.weight", l); L.wi = add(b, f, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.2.DenseReluDense.wo.weight", l); L.wo = add(b, d, f, 0);
  }
  for (int l = 0; l < c.n_dec_layers; ++l) {
    snprintf(b, sizeof b, "decoder.block.%d.layer.1.EncDecAttention.k.weight", l);
    const size_t o = add(b, d, d, 0);
    if (l == 0) e.o_ckv = o;
    snprintf(b, sizeof b, "decoder.block.%d.layer.1.EncDecAttention.v.weight", l); add(b, d, d, 0);
  }
  for (int l = 0; l < c.n_enc_layers; ++l) {
    EncLayer& L = e.enc[l];
    snprintf(b, sizeof b, "encoder.block.%d.layer.0.SelfAttention.q.weight", l); L.qkv = add(b, d, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.0.SelfAttention.k.weight", l); add(b, d, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.0.SelfAttention.v.weight", l); add(b, d, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.0.SelfAttention.o.weight", l); L.o = add(b, d, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.1.DenseReluDense.wi.weight", l); L.wi = add(b, f, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.1.DenseReluDense.wo.weight", l); L.wo = add(b, d, f, 0);
  }
  e.o_Wf = add("encoder.visual_embedding.feat_embedding.0.weight", d, c.feat_dim, 0);
  // (2) the tail: everything a kernel reads in fp32 (embedding table, norm weights, the small visual parameters, biases,
  //     relative-position tables). With N > 1 GPUs it is all-reduced and updated by every rank, so the fp32 masters of
  //     this region are always current everywhere; only region (1) is ever sharded.
  off = align_up(off, 64);
  e.o_tail = off;
  e.o_shared = add("shared.weight", c.vocab_size, d, 0);
  for (int l = 0; l < c.n_dec_layers; ++l) {
    DecLayer& L = e.dec[l];
    snprintf(b, sizeof b, "decoder.block.%d.layer.0.layer_norm.weight", l); L.ln0 = add(b, 1, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.1.layer_norm.weight", l); L.ln1 = add(b, 1, d, 0);
    snprintf(b, sizeof b, "decoder.block.%d.layer.2.layer_norm.weight", l); L.ln2 = add(b, 1, d, 0);
  }
  e.o_dec_final = add("decoder.final_layer_norm.weight", 1, d, 0);
  for (int l = 0; l < c.n_enc_layers; ++l) {
    EncLayer& L = e.enc[l];
    snprintf(b, sizeof b, "encoder.block.%d.layer.0.layer_norm.weight", l); L.ln0 = add(b, 1, d, 0);
    snprintf(b, sizeof b, "encoder.block.%d.layer.1.layer_norm.weight", l); L.ln1 = add(b, 1, d, 0);
  }
  e.o_enc_final = add("encoder.final_layer_norm.weight", 1, d, 0);
  e.o_wf = add("encoder.visual_embedding.feat_embedding.1.weight", 1, d, 0);
  e.o_Wp = add("encoder.visual_embedding.absolute_vis_pos_embedding.0.weight", d, 5, 0);
  e.o_wp = add("encoder.visual_embedding.absolute_vis_pos_embedding.1.weight", 1, d, 0);
  e.o_img = add("encoder.visual_embedding.img_order_embedding.weight", c.n_images, d, 0);
  off = align_up(off, 64);
  e.n_decay = off;
  // ---- no-decay group: names containing "bias" (trainer_base.py:148-160) ----------------------------------
  e.o_bf = add("encoder.visual_embedding.feat_embedding.0.bias", 1, d, 1);
  e.o_bp = add("encoder.visual_embedding.absolute_vis_pos_embedding.0.bias", 1, d, 1);
  e.o_enc_rel = add("encoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight", c.n_buckets, c.n_heads, 1);
  e.o_dec_rel = add("decoder.block.0.layer.0.SelfAttention.relative_attention_bias.weight", c.n_buckets, c.n_heads, 1);
  off = align_up(off, 64);
  e.n_train = off;
  // ---- never receive a gradient (modeling_t5_our.py:379-380 are unused) -------------------------------------
  add("prototype_fc1.weight", d, d, 2);
  add("prototype_fc1.bias", 1, d, 2);
  add("prototype_fc2.weight", d, d, 2);
  add("prototype_fc2.bias", 1, d, 2);
  off = align_up(off, 64);
  e.n_total = off;
  // q,k,v of one layer must be adjacent (no alignment gap): d*d is a multiple of 64
  VQ_CHECK(((size_t)d * d) % 64 == 0, "engine: d*d must be a multiple of 64");
  return 0;
}

// --------------------------------------------------------------------------------------------------- workspace
struct Bump {
  uint8_t* base;
  int64_t off = 0;
  std::map<std::string, int64_t>* names;
  template <typename Tp>
  Tp* take(size_t count, const char* name = nullptr) {
    off = (off + 255) / 256 * 256;
    Tp* p = base ? reinterpret_cast<Tp*>(base + off) : nullptr;
    if (name && names) (*names)[name] = off;
    off += (int64_t)(count * sizeof(Tp));
    return p;
  }
};

int64_t engine_carve(Engine& e, uint8_t* base, int B, int L, int N, int T) {
  const vqacl_config& c = e.cfg;
  const int d = c.d_model, f = c.d_ff, H = c.n_heads;
  const int S = L + N, S2 = S + 2;
  const size_t M = (size_t)B * S, Md = (size_t)B * T, M2 = (size_t)B * S2;
  const size_t fw = (size_t)(f + 31) / 32;   // ReLU bitmask words per row
  const int Le = c.n_enc_layers, Ld = c.n_dec_layers;
  Workspace w;
  std::map<std::string, int64_t> names;
  Bump bp{base, 0, &names};
  const int ldv = (c.vocab_size + 255) / 256 * 256;
  w.feats_bf16 = bp.take<bf16>((size_t)B * N * c.feat_dim);
  w.featpre = bp.take<float>((size_t)B * N * d);
  w.x.resize(2 * Le + 1);
  for (auto& p : w.x) p = bp.take<float>(M * d);
  w.n1.resize(Le); w.qkv.resize(Le); w.ao.resize(Le); w.n2.resize(Le); w.h.resize(Le); w.hmask.resize(Le); w.lse_e.resize(Le);
  for (int l = 0; l < Le; ++l) {
    w.n1[l] = bp.take<bf16>(M * d);
    w.qkv[l] = bp.take<bf16>(M * 3 * d);
    w.ao[l] = bp.take<bf16>(M * d);
    w.n2[l] = bp.take<bf16>(M * d);
    w.h[l] = bp.take<bf16>(M * f);
    w.hmask[l] = bp.take<uint32_t>(M * fw);
    w.lse_e[l] = bp.take<float>((size_t)B * H * S);
  }
  w.enc_hidden = bp.take<float>(M * d, "encoder_hidden_states");
  w.mem = bp.take<bf16>(M2 * d, "decoder_memory");
  w.enc_mask = bp.take<float>((size_t)B * S);
  w.cross_mask = bp.take<float>((size_t)B * S2, "cross_mask");
  w.mask01 = bp.take<float>((size_t)B * S2, "encoder_attention_mask");
  w.meanQ = bp.take<float>((size_t)B * d, "meanQ");
  w.meanV = bp.take<float>((size_t)B * d, "meanV");
  w.curQ = bp.take<float>((size_t)c.n_ques * d, "curQ");
  w.curV = bp.take<float>((size_t)c.n_cate * d, "curV");
  w.cntQ = bp.take<float>(c.n_ques, "cntQ");
  w.cntV = bp.take<float>(c.n_cate, "cntV");
  w.pnorm = bp.take<float>((size_t)(c.n_ques > c.n_cate ? c.n_ques : c.n_cate) * d);
  w.memdQ = bp.take<float>((size_t)B * d);
  w.memdV = bp.take<float>((size_t)B * d);
  w.mem_ssq = bp.take<float>((size_t)2 * B);
  w.mem_loss = bp.take<float>(4, "loss_memory");
  w.idxQ = bp.take<int64_t>(B, "idxQ");
  w.idxV = bp.take<int64_t>(B, "idxV");
  w.dec_ids = bp.take<int64_t>(Md, "decoder_input_ids");
  w.y.resize(3 * Ld + 1);
  for (auto& p : w.y) p = bp.take<float>(Md * d);
  w.dn1.resize(Ld); w.dqkv.resize(Ld); w.dao.resize(Ld); w.dn2.resize(Ld); w.cq.resize(Ld); w.cao.resize(Ld); w.dn3.resize(Ld);
  w.dh.resize(Ld); w.dhmask.resize(Ld); w.lse_s.resize(Ld); w.lse_c.resize(Ld);
  for (int l = 0; l < Ld; ++l) {
    w.dn1[l] = bp.take<bf16>(Md * d);
    w.dqkv[l] = bp.take<bf16>(Md * 3 * d);
    w.dao[l] = bp.take<bf16>(Md * d);
    w.dn2[l] = bp.take<bf16>(Md * d);
    w.cq[l] = bp.take<bf16>(Md * d);
    w.cao[l] = bp.take<bf16>(Md * d);
    w.dn3[l] = bp.take<bf16>(Md * d);
    w.dh[l] = bp.take<bf16>(Md * f);
    w.dhmask[l] = bp.take<uint32_t>(Md * fw);
    w.lse_s[l] = bp.take<float>((size_t)B * H * T);
    w.lse_c[l] = bp.take<float>((size_t)B * H * T);
  }
  w.kv_all = bp.take<bf16>(M2 * (size_t)Ld * 2 * d);
  w.yfin = bp.take<bf16>(Md * d);
  w.logits = bp.take<bf16>(Md * (size_t)ldv, "logits");
  w.lse_ce = bp.take<float>(Md);
  w.loss_rows = bp.take<float>(Md, "loss_rows");
  w.w_rows = bp.take<float>(Md, "w_rows");
  w.loss = bp.take<float>(4, "loss");
  // backward
  w.gd = bp.take<float>(Md * d);
  for (auto& p : w.gdb_ring) p = bp.take<bf16>(Md * d);
  w.t_d768 = bp.take<bf16>(Md * d);
  w.t_d768_f32 = bp.take<float>(Md * d);
  w.t_parts = bp.take<float>((size_t)3 * Md * d);
  for (int i = 0; i < Workspace::RING; ++i) {
    w.t_dqkv[i] = bp.take<bf16>(Md * 3 * d);
    w.t_dh[i] = bp.take<bf16>(Md * f);
    w.t_dcq[i] = bp.take<bf16>(Md * d);
  }
  w.ge = bp.take<float>(M * d);
  for (auto& p : w.geb_ring) p = bp.take<bf16>(M * d);
  w.t_e768 = bp.take<bf16>(M * d);
  for (int i = 0; i < Workspace::RING; ++i) {
    w.t_eqkv[i] = bp.take<bf16>(M * 3 * d);
    w.t_eh[i] = bp.take<bf16>(M * f);
  }
  w.dkv_all = bp.take<bf16>(M2 * (size_t)Ld * 2 * d);
  w.dmem = bp.take<bf16>(M2 * d);
  w.dfeatpre = bp.take<bf16>((size_t)B * N * d);
  w.vis_partials = bp.take<float>((size_t)num_sms() * 10 * d);
  const int64_t total = (bp.off + 255) / 256 * 256;
  if (base) {
    e.w = w;
    e.ws_names = names;
    e.ws_base = base;
    e.ws_bytes = total;
    e.B = B; e.L = L; e.N = N; e.T = T;
    e.ldv = ldv;
    e.fwd_valid = false;
  }
  return total;
}

// --------------------------------------------------------------------------------------------------- GEMM helpers
// SMs the decoder's weight-gradient GEMMs (side stream) may occupy while the latency-bound dX / attention / norm chain runs on
// the main stream. Default 0 = no limit: 48 / 64 / 96 SMs measured 2.69 / 2.42 / 2.34 ms for the decoder-layer backward against
// 2.36-2.40 ms unlimited (the side stream then falls behind and the chain waits for it at the two-layer lag) — kept as a switch
static int g_dec_dw_sms = [] { const char* ev = getenv("VQACL_DEC_DW_SMS"); return ev ? atoi(ev) : 0; }();
// split-K factor of the decoder's deep dX GEMMs (wi: K = d_ff, qkv: K = 3 d) into an fp32 buffer the RMSNorm backward reads and
// clears (VQACL_DEC_DX_SPLITS=1: single-pass bf16). Three slices make the two GEMMs 2x faster alone (126 instead of 42 CTAs
// streaming operands). Measured twice: with six separate dW launches on the side stream the step got 0.1-0.2 ms SLOWER (the
// wide dX launches and the dW launches fought for SMs); with the dW GEMMs grouped into one launch per layer the decoder-layer
// backward drops from 2.22-2.25 to 2.10-2.14 ms
// the decoder's six weight gradients of a layer as ONE grouped launch at the end of the layer (VQACL_DEC_DW_GROUPED=0: one launch
// each, right after the kernel that produced its dY)
static int g_dec_dw_grouped = [] { const char* ev = getenv("VQACL_DEC_DW_GROUPED"); return (ev && ev[0] == '0') ? 0 : 1; }();
static int g_dec_dx_splits = [] { const char* ev = getenv("VQACL_DEC_DX_SPLITS"); return ev && atoi(ev) > 0 ? atoi(ev) : 3; }();
// dX[rows, n_in] = dY[rows, n_out] * W[n_out, n_in]      (W stored row-major -> MN-major B operand)
static int gemm_dx(const bf16* dY, int lddy, const bf16* Wt, int n_out, int n_in, void* C, int ldc, int rows, int epi, cudaStream_t st,
                   const void* R = nullptr, int ldr = 0, float alpha = 1.f, int splits = 1) {
  GemmArgs g{};
  g.epi = epi; g.M = rows; g.N = n_in; g.K = n_out; g.C = C; g.ldc = ldc; g.R = R; g.ldr = ldr; g.alpha = alpha; g.splits = splits;
  return gemm_bf16(GemmOperand{dY, lddy, false}, GemmOperand{Wt, n_in, true}, g, 0, st);
}
// dW[n_out, n_in] += dY[rows, n_out]^T * X[rows, n_in]    (both operands MN-major, split-K over rows, fp32 red.add)
static int gemm_dw(const bf16* dY, int lddy, const bf16* X, int ldx, float* dWt, int n_out, int n_in, int rows, cudaStream_t st,
                   int sm_limit = 0) {
  GemmArgs g{};
  g.epi = EPI_ATOMIC_F32; g.M = n_out; g.N = n_in; g.K = rows; g.C = dWt; g.ldc = n_in; g.alpha = 1.f; g.sm_limit = sm_limit;
  const int tiles = ((n_out + 127) / 128) * ((n_in + 255) / 256);
  const int kblocks = (rows + 63) / 64;
  int splits = (2 * num_sms()) / (tiles > 0 ? tiles : 1);
  if (splits > kblocks / 8) splits = kblocks / 8;
  if (splits < 1) splits = 1;
  g.splits = splits;
  return gemm_bf16(GemmOperand{dY, lddy, true}, GemmOperand{X, ldx, true}, g, 0, st);
}


// --------------------------------------------------------------------------------------------------- forward
int check_batch(const Engine& e, const vqacl_batch* b, bool need_labels) {
  VQ_CHECK(e.P && e.W, "engine: parameter arena not bound");
  VQ_CHECK(e.ws_base, "engine: workspace not bound");
  VQ_CHECK(e.enc_bucket && e.dec_bucket, "engine: relative-position bucket maps not set");
  VQ_CHECK(b->B == e.B && b->L == e.L && b->N == e.N && (!need_labels || b->T == e.T),
           "engine: batch shape (B=%d L=%d N=%d T=%d) does not match the bound workspace (B=%d L=%d N=%d T=%d)", b->B, b->L,
           b->N, b->T, e.B, e.L, e.N, e.T);
  // the decoder attends to the encoder output plus the two retrieved prototype rows: L + N + 2 keys. Up to 64 keys run on the
  // single-tile attention kernels, longer visual sequences (configs[3]) on the generic multi-tile ones (<= 256 keys).
  VQ_CHECK(b->L + b->N + 2 <= 256 && b->L >= 1 && b->N >= 1, "engine: encoder length L+N=%d must be in [2,254]", b->L + b->N);
  VQ_CHECK(b->L <= 64, "engine: text width L=%d must be at most 64 (the relative-position bias corner must fit one attention tile)", b->L);
  VQ_CHECK(!need_labels || (b->T >= 1 && b->T <= 64), "engine: target width T=%d must be in [1,64]", b->T);
  VQ_CHECK((b->vis_feats || b->vis_feats_bf16) && b->boxes && b->input_ids, "engine: missing batch pointers");
  return 0;
}

int encoder_forward(Engine& e, const vqacl_batch* b, cudaStream_t st) {
  const vqacl_config& c = e.cfg;
  Workspace& w = e.w;
  const int d = c.d_model, f = c.d_ff, H = c.n_heads;
  const int B = b->B, L = b->L, N = b->N, S = L + N, S2 = S + 2;
  const int M = B * S;
  VQ_TRY(wait_params(e, 0, st));   // embeddings + visual projection + final norms
  VQ_TRY(build_keymasks(b->input_ids, B, L, S, c.pad_id, w.enc_mask, w.cross_mask, w.mask01, st));
  // embeddings: text rows [0,L), visual rows [L,S)   (modeling_t5_our.py:196-214, :247)
  VQ_TRY(embed_fwd(b->input_ids, B, L, e.P + e.o_shared, w.x[0], S, 0, e.drop(SITE_ENC_EMB), c.vocab_size, e.err_flags(), st));
  // RoI features: fp32 from the reference's collate_fn (cast once) or already bf16 from a packed feature shard
  const bf16* feats = reinterpret_cast<const bf16*>(b->vis_feats_bf16);
  if (!feats) {
    VQ_TRY(cast_f32_to_bf16(b->vis_feats, w.feats_bf16, (size_t)B * N * c.feat_dim, st));
    feats = w.feats_bf16;
  }
  if (gemm_vis_tail_on() && B * N >= 192) {
    // VisualEmbedding.forward (modeling_t5_our.py:93-143) in ONE launch: the 2048 -> 768 projection on tcgen05 (TMA-staged), and —
    // as the row tail of the CTA pair that owns a 256-row block — bias + RMSNorm, the 5 -> 768 box projection + RMSNorm, the
    // image / object order embeddings and the embedding dropout, written straight into rows [L, S) of the residual stream.
    // featpre (fp32) is still written: the backward re-reads it.
    const Dropout dr = e.drop(SITE_ENC_EMB);
    GemmArgs g{};
    g.epi = EPI_F32; g.M = B * N; g.N = d; g.K = c.feat_dim; g.C = w.featpre; g.ldc = d; g.alpha = 1.f; g.splits = 1;
    g.tail = 2; g.tail_eps = c.eps;
    g.vt.boxes = b->boxes; g.vt.bf = e.P + e.o_bf; g.vt.wf = e.P + e.o_wf; g.vt.Wp = e.P + e.o_Wp; g.vt.bp = e.P + e.o_bp;
    g.vt.wp = e.P + e.o_wp; g.vt.img_emb = e.P + e.o_img; g.vt.shared = e.P + e.o_shared; g.vt.x = w.x[0];
    g.vt.V = c.vocab_size; g.vt.N = N; g.vt.S = S; g.vt.L = L;
    g.vt.drop_thr = dr.thr; g.vt.drop_inv_keep = dr.inv_keep; g.vt.drop_seed = dr.seed;
    VQ_TRY(gemm_bf16(GemmOperand{feats, c.feat_dim, false}, GemmOperand{e.W + e.o_Wf, c.feat_dim, false}, g, 0, st));
  } else {
    VQ_TRY(gemm_fwd(feats, c.feat_dim, e.W + e.o_Wf, c.feat_dim, w.featpre, d, B * N, d, EPI_F32, st));
    VisArgs va{};
    va.featpre = w.featpre; va.boxes = b->boxes; va.bf = e.P + e.o_bf; va.wf = e.P + e.o_wf; va.Wp = e.P + e.o_Wp;
    va.bp = e.P + e.o_bp; va.wp = e.P + e.o_wp; va.img_emb = e.P + e.o_img; va.shared = e.P + e.o_shared;
    va.V = c.vocab_size; va.B = B; va.N = N; va.S = S; va.L = L; va.eps = c.eps; va.x = w.x[0]; va.drop = e.drop(SITE_ENC_EMB);
    VQ_TRY(vis_embed_fwd(va, st));
  }
  // The RMSNorm that opens a sub-layer is folded into the residual GEMM that closes the previous one (row tail of the CTA-pair
  // kernel: the pair that wrote a 256-row block normalises it while it is still in L2) whenever the blocks fill the machine
  // as well as the tiles would; otherwise (and for the first layer, which follows the embeddings) it is its own kernel.
  const bool fold = gemm_row_tail_ok(M);
  auto gemm_resid_norm = [&](const bf16* A, int lda, const bf16* Wt, int K, float* C, const float* R, Dropout dr, const float* nw, bf16* nout) -> int {
    GemmArgs g{};
    g.epi = EPI_RESID_F32; g.M = M; g.N = d; g.K = K; g.C = C; g.ldc = d; g.R = R; g.ldr = d; g.alpha = 1.f; g.splits = 1;
    g.drop_thr = dr.thr; g.drop_inv_keep = dr.inv_keep; g.seed = dr.seed; g.site = dr.site;
    g.tail = 1; g.tail_w = nw; g.tail_out = nout; g.tail_ld = d; g.tail_eps = c.eps;
    return gemm_bf16(GemmOperand{A, lda, false}, GemmOperand{Wt, K, false}, g, 0, st);
  };
  for (int l = 0; l < c.n_enc_layers; ++l) {
    const EncLayer& P = e.enc[l];
    VQ_TRY(wait_params(e, 1 + l, st));
    RmsFwdArgs r{};
    r.x = w.x[2 * l]; r.w = e.P + P.ln0; r.y_bf16 = w.n1[l]; r.ld_bf16 = d; r.M = M; r.eps = c.eps; r.scale = 1.f;
    if (!fold || l == 0) VQ_TRY(rmsnorm_fwd(r, st));
    VQ_TRY(gemm_fwd(w.n1[l], d, e.W + P.qkv, d, w.qkv[l], 3 * d, M, 3 * d, EPI_BF16, st));
    AttnArgs a{};
    a.q = w.qkv[l]; a.k = w.qkv[l] + d; a.v = w.qkv[l] + 2 * d; a.ldq = a.ldk = a.ldv = 3 * d;
    a.o = w.ao[l]; a.ldo = d; a.lse = w.lse_e[l]; a.B = B; a.H = H; a.Sq = S; a.Sk = S;
    a.rel_table = e.P + e.o_enc_rel; a.rel_bucket = e.enc_bucket; a.rel_mode = 1; a.Lt = L; a.keymask = w.enc_mask; a.causal = 0;
    const Dropout dp = e.drop(site_enc(l, 0));
    a.drop_thr = dp.thr; a.drop_inv_keep = dp.inv_keep; a.seed = dp.seed; a.site = dp.site;
    VQ_TRY(attn_fwd(a, st));
    if (fold) {
      VQ_TRY(gemm_resid_norm(w.ao[l], d, e.W + P.o, d, w.x[2 * l + 1], w.x[2 * l], e.drop(site_enc(l, 1)), e.P + P.ln1, w.n2[l]));
    } else {
      VQ_TRY(gemm_fwd(w.ao[l], d, e.W + P.o, d, w.x[2 * l + 1], d, M, d, EPI_RESID_F32, st, w.x[2 * l], d, e.drop(site_enc(l, 1))));
      r.x = w.x[2 * l + 1]; r.w = e.P + P.ln1; r.y_bf16 = w.n2[l];
      VQ_TRY(rmsnorm_fwd(r, st));
    }
    VQ_TRY(gemm_fwd(w.n2[l], d, e.W + P.wi, d, w.h[l], f, M, f, EPI_RELU_BF16, st, w.hmask[l], (f + 31) / 32, e.drop(site_enc(l, 2))));
    if (fold && l + 1 < c.n_enc_layers) {     // + the first norm of the next layer
      VQ_TRY(gemm_resid_norm(w.h[l], f, e.W + P.wo, f, w.x[2 * l + 2], w.x[2 * l + 1], e.drop(site_enc(l, 3)), e.P + e.enc[l + 1].ln0, w.n1[l + 1]));
    } else {
      VQ_TRY(gemm_fwd(w.h[l], f, e.W + P.wo, f, w.x[2 * l + 2], d, M, d, EPI_RESID_F32, st, w.x[2 * l + 1], d, e.drop(site_enc(l, 3))));
    }
  }
  // final norm + dropout (:314-315): fp32 copy for the SI path / caller, bf16 straight into the [B,S+2,d] decoder memory
  RmsFwdArgs r{};
  r.x = w.x[2 * c.n_enc_layers]; r.w = e.P + e.o_enc_final; r.y_bf16 = w.mem; r.ld_bf16 = d; r.y_f32 = w.enc_hidden; r.ld_f32 = d;
  r.M = M; r.eps = c.eps; r.scale = 1.f; r.in_rpb = S; r.out_rpb = S2; r.drop = e.drop(SITE_ENC_FINAL);
  VQ_TRY(rmsnorm_fwd(r, st));
  // SI path, part 1: token means (+ per-class sums for the update)   (:585-588, :601-611)
  VQ_TRY(proto_means(w.enc_hidden, B, S, c.split_L, w.meanQ, w.meanV, st));
  return 0;
}

int si_path(Engine& e, const vqacl_batch* b, const vqacl_proto_state* ps, bool sums_ready, cudaStream_t st) {
  const vqacl_config& c = e.cfg;
  Workspace& w = e.w;
  const int B = b->B, S2 = b->L + b->N + 2, S = b->L + b->N;
  VQ_CHECK(ps && ps->Q_prototype && ps->V_prototype, "engine: prototype banks missing (Q_prototype / V_prototype)");
  e.mem_loss_valid = false;
  if (ps->proto_update) {
    VQ_CHECK(b->cate_labels && b->ques_labels, "engine: proto_update needs cate_labels and ques_labels");
    VQ_CHECK(ps->Q_num && ps->V_num, "engine: proto_update needs the count buffers");
    if (ps->memory_loss) {
      // modeling_t5_our.py:590-592: against the banks as the PREVIOUS step left them (the update follows at :597)
      VQ_TRY(proto_memory_loss(w.meanQ, w.meanV, b->ques_labels, b->cate_labels, ps->Q_prototype, ps->V_prototype, c.n_ques, c.n_cate, B,
                               w.memdQ, w.memdV, w.mem_ssq, w.mem_loss, st));
      e.mem_loss_valid = true;
    }
    if (!sums_ready) {
      VQ_TRY(proto_scatter_mean(w.meanQ, b->ques_labels, B, c.n_ques, w.curQ, w.cntQ, st));
      VQ_TRY(proto_scatter_mean(w.meanV, b->cate_labels, B, c.n_cate, w.curV, w.cntV, st));
    } else {
      VQ_TRY(proto_div(w.curQ, w.cntQ, c.n_ques, st));
      VQ_TRY(proto_div(w.curV, w.cntV, c.n_cate, st));
    }
    ProtoUpdateArgs u{};
    u.curQ = w.curQ; u.curV = w.curV; u.cntQ = w.cntQ; u.cntV = w.cntV;
    u.Qproto = ps->Q_prototype; u.Vproto = ps->V_prototype; u.numQ = ps->Q_num; u.numV = ps->V_num;
    u.CQ = c.n_ques; u.CV = c.n_cate; u.task_id = ps->task_id; u.first_step_of_task = ps->first_step_of_task;
    u.has_mem = ps->has_mem; u.alpha = ps->alpha; u.beta = ps->beta;
    VQ_TRY(proto_update(u, st));
  }
  // retrieval + feature mix (:601-615): rows S and S+1 of the decoder memory
  VQ_TRY(proto_retrieve(ps->Q_prototype, c.n_ques, w.meanQ, B, w.mem, S2, S, w.idxQ, nullptr, w.pnorm, st));
  VQ_TRY(proto_retrieve(ps->V_prototype, c.n_cate, w.meanV, B, w.mem, S2, S + 1, w.idxV, nullptr, w.pnorm, st));
  return 0;
}

static int ensure_side_stream(Engine& e);

static int decoder_forward(Engine& e, const vqacl_batch* b, cudaStream_t st) {
  const vqacl_config& c = e.cfg;
  Workspace& w = e.w;
  const int d = c.d_model, f = c.d_ff, H = c.n_heads, Ld = c.n_dec_layers;
  const int B = b->B, T = b->T, S2 = b->L + b->N + 2;
  const int Md = B * T, M2 = B * S2;
  const int ldkv = Ld * 2 * d;
  VQ_TRY(wait_params(e, 1 + c.n_enc_layers, st));   // decoder + cross-KV weights (last optimizer chunk)
  e.g_prezeroed = false;
  if (e.prezero_request && e.G) {
    // From here on nothing reads the previous step's gradients any more (the optimizer is ordered before this point): clear
    // the arena for the coming backward on the side stream, hidden behind the decoder forward (0.9 GB, ~0.14 ms of HBM time)
    VQ_TRY(ensure_side_stream(e));
    VQ_CUDA(cudaEventRecord(e.ev_fork, st));
    VQ_CUDA(cudaStreamWaitEvent(e.side, e.ev_fork, 0));
    VQ_CUDA(cudaMemsetAsync(e.G, 0, e.n_train * sizeof(float), e.side));
    VQ_CUDA(cudaEventRecord(e.ev_gzero, e.side));
    e.g_prezeroed = true;
  }
  if (b->decoder_input_ids) {                                                                      // :617-629 (given explicitly)
    VQ_CUDA(cudaMemcpyAsync(w.dec_ids, b->decoder_input_ids, (size_t)Md * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
  } else {
    VQ_TRY(shift_right(b->labels, w.dec_ids, B, T, c.start_id, c.pad_id, st));                    // :620
  }
  VQ_TRY(embed_fwd(w.dec_ids, B, T, e.P + e.o_shared, w.y[0], T, 0, e.drop(SITE_DEC_EMB), c.vocab_size, e.err_flags(), st));
  // cross-attention K/V of every decoder layer in one GEMM over the decoder memory
  VQ_TRY(gemm_fwd(w.mem, d, e.W + e.o_ckv, d, w.kv_all, ldkv, M2, ldkv, EPI_BF16, st));
  // FFN-out (K = d_ff = 3072 against 39-78 output tiles at M = B*T rows) as a 3-way split-K: three times the CTAs stream the
  // operands (a CTA's stream is bound by its SM's L2 port: 17.9 -> ~9 us), each slice stores an fp32 slab, and the NEXT norm
  // kernel forms y[3l+3] = y[3l+2] + dropout(slab0 + slab1 + slab2) in that fixed order before normalising — deterministic,
  // unlike an atomic meeting point. VQACL_DEC_FFN_SPLITS=1 restores the single-pass residual epilogue.
  static const int fsplit_req = [] { const char* ev = getenv("VQACL_DEC_FFN_SPLITS"); const int v = ev ? atoi(ev) : 3; return v >= 1 && v <= 3 ? v : 3; }();
  // the slab count the GEMM will really use (gemm_bf16 never leaves a K slice empty): the norm kernel must add exactly those
  const int fsplit = gemm_split_count(f, fsplit_req);
  auto ffn_out_pending = [&](RmsFwdArgs& r, int l_prev) {     // make r's norm consume the slabs of layer l_prev's FFN-out GEMM
    r.parts = w.t_parts; r.n_parts = fsplit; r.part_stride = (long long)Md * d;
    r.resid = w.y[3 * l_prev + 2]; r.x_out = w.y[3 * l_prev + 3]; r.resid_drop = e.drop(site_dec(l_prev, 5));
  };
  for (int l = 0; l < Ld; ++l) {
    const DecLayer& P = e.dec[l];
    RmsFwdArgs r{};
    r.x = w.y[3 * l]; r.w = e.P + P.ln0; r.y_bf16 = w.dn1[l]; r.ld_bf16 = d; r.M = Md; r.eps = c.eps; r.scale = 1.f;
    if (fsplit > 1 && l > 0) ffn_out_pending(r, l - 1);
    VQ_TRY(rmsnorm_fwd(r, st));
    r.parts = nullptr;
    VQ_TRY(gemm_fwd(w.dn1[l], d, e.W + P.qkv, d, w.dqkv[l], 3 * d, Md, 3 * d, EPI_BF16, st));
    AttnArgs a{};
    a.q = w.dqkv[l]; a.k = w.dqkv[l] + d; a.v = w.dqkv[l] + 2 * d; a.ldq = a.ldk = a.ldv = 3 * d;
    a.o = w.dao[l]; a.ldo = d; a.lse = w.lse_s[l]; a.B = B; a.H = H; a.Sq = T; a.Sk = T;
    a.rel_table = e.P + e.o_dec_rel; a.rel_bucket = e.dec_bucket; a.rel_mode = 2; a.keymask = nullptr; a.causal = 1;
    Dropout dp = e.drop(site_dec(l, 0));
    a.drop_thr = dp.thr; a.drop_inv_keep = dp.inv_keep; a.seed = dp.seed; a.site = dp.site;
    VQ_TRY(attn_fwd(a, st));
    VQ_TRY(gemm_fwd(w.dao[l], d, e.W + P.o, d, w.y[3 * l + 1], d, Md, d, EPI_RESID_F32, st, w.y[3 * l], d, e.drop(site_dec(l, 1))));
    // cross attention to the [B,S+2,d] memory: zero position bias, (1-mask)*-1e9 on text pads
    r.x = w.y[3 * l + 1]; r.w = e.P + P.ln1; r.y_bf16 = w.dn2[l];
    VQ_TRY(rmsnorm_fwd(r, st));
    VQ_TRY(gemm_fwd(w.dn2[l], d, e.W + P.cq, d, w.cq[l], d, Md, d, EPI_BF16, st));
    AttnArgs x{};
    x.q = w.cq[l]; x.ldq = d; x.k = w.kv_all + (size_t)l * 2 * d; x.v = x.k + d; x.ldk = x.ldv = ldkv;
    x.o = w.cao[l]; x.ldo = d; x.lse = w.lse_c[l]; x.B = B; x.H = H; x.Sq = T; x.Sk = S2;
    x.rel_mode = 0; x.keymask = w.cross_mask; x.causal = 0;
    dp = e.drop(site_dec(l, 2));
    x.drop_thr = dp.thr; x.drop_inv_keep = dp.inv_keep; x.seed = dp.seed; x.site = dp.site;
    VQ_TRY(attn_fwd(x, st));
    VQ_TRY(gemm_fwd(w.cao[l], d, e.W + P.co, d, w.y[3 * l + 2], d, Md, d, EPI_RESID_F32, st, w.y[3 * l + 1], d, e.drop(site_dec(l, 3))));
    r.x = w.y[3 * l + 2]; r.w = e.P + P.ln2; r.y_bf16 = w.dn3[l];
    VQ_TRY(rmsnorm_fwd(r, st));
    VQ_TRY(gemm_fwd(w.dn3[l], d, e.W + P.wi, d, w.dh[l], f, Md, f, EPI_RELU_BF16, st, w.dhmask[l], (f + 31) / 32, e.drop(site_dec(l, 4))));
    if (fsplit > 1) {
      GemmArgs g{};
      g.epi = EPI_F32; g.M = Md; g.N = d; g.K = f; g.C = w.t_parts; g.ldc = d; g.alpha = 1.f; g.splits = fsplit;
      g.split_stride = (long long)Md * d;
      VQ_TRY(gemm_bf16(GemmOperand{w.dh[l], f, false}, GemmOperand{e.W + P.wo, f, false}, g, 0, st));
    } else {
      VQ_TRY(gemm_fwd(w.dh[l], f, e.W + P.wo, f, w.y[3 * l + 3], d, Md, d, EPI_RESID_F32, st, w.y[3 * l + 2], d, e.drop(site_dec(l, 5))));
    }
  }
  // final norm, dropout, x d^-1/2 (:666), tied LM head (:671), CE with reduction='none' (:683-686)
  RmsFwdArgs r{};
  r.x = w.y[3 * Ld]; r.w = e.P + e.o_dec_final; r.y_bf16 = w.yfin; r.ld_bf16 = d; r.M = Md; r.eps = c.eps;
  r.scale = 1.f / sqrtf((float)d); r.drop = e.drop(SITE_DEC_FINAL);
  if (fsplit > 1) ffn_out_pending(r, Ld - 1);
  VQ_TRY(rmsnorm_fwd(r, st));
  VQ_TRY(gemm_fwd(w.yfin, d, e.W + e.o_shared, d, w.logits, e.ldv, Md, c.vocab_size, EPI_BF16, st));
  if (b->labels) VQ_TRY(ce_fwd(w.logits, e.ldv, Md, c.vocab_size, b->labels, w.lse_ce, w.loss_rows, st));
  return 0;
}

// --------------------------------------------------------------------------------------------------- backward
struct SavedBatch {
  vqacl_batch b;
  bool valid = false;
};
static std::map<Engine*, SavedBatch> g_saved;

// Backward runs in stages so that the host can start the gradient all-reduce of a finished arena range while later
// stages still compute (SURVEY.md §8e):
//   stage 0            : CE + LM head + decoder final norm
//   stage 1 .. Ld      : decoder layer Ld - stage
//   stage Ld+1         : decoder token embedding, cross-attention K/V projection (all layers), encoder final norm
//   stage Ld+2 .. Ld+1+Le : encoder layer Le - (stage - Ld - 1)
//   stage Ld+Le+2      : text / visual embeddings
static int n_backward_stages(const Engine& e) { return e.cfg.n_dec_layers + e.cfg.n_enc_layers + 3; }

// arena range [*a, *b) whose gradients are final once `stage` has run (possibly empty). The tail region (embedding table,
// norm weights, small visual parameters, biases: [o_tail, n_train)) collects contributions from every stage and is final
// only after the last one, where it is reported together with the visual projection.
static void backward_stage_range(const Engine& e, int stage, int64_t* a, int64_t* b) {
  const int Ld = e.cfg.n_dec_layers, Le = e.cfg.n_enc_layers;
  *a = *b = 0;
  if (stage >= 1 && stage <= Ld) {
    const int l = Ld - stage;
    *a = (int64_t)e.dec[l].qkv;
    *b = (int64_t)(l + 1 < Ld ? e.dec[l + 1].qkv : e.o_ckv);
  } else if (stage == Ld + 1) {
    *a = (int64_t)e.o_ckv;
    *b = (int64_t)(Le > 0 ? e.enc[0].qkv : e.o_Wf);
  } else if (stage >= Ld + 2 && stage <= Ld + 1 + Le) {
    const int l = Le - (stage - Ld - 1);
    *a = (int64_t)e.enc[l].qkv;
    *b = (int64_t)(l + 1 < Le ? e.enc[l + 1].qkv : e.o_Wf);
  } else if (stage == Ld + Le + 2) {
    *a = (int64_t)e.o_Wf;
    *b = (int64_t)e.n_train;
  }
}

int wait_params(Engine& e, int chunk, cudaStream_t st) {
  if (e.ext_pending) {   // sharded optimizer: the host all-gathers refreshed bf16 weights on its communication stream
    VQ_CHECK(chunk >= 0 && chunk < (int)e.ext_ev.size(), "wait_params: chunk %d out of range", chunk);
    if (e.ext_ev[chunk]) VQ_CUDA(cudaStreamWaitEvent(st, e.ext_ev[chunk], 0));
    if (chunk + 1 == (int)e.ext_ev.size()) e.ext_pending = false;
  }
  if (!e.opt_pending) return 0;
  VQ_CHECK(chunk >= 0 && chunk < (int)e.ev_opt.size(), "wait_params: chunk %d out of range", chunk);
  VQ_CUDA(cudaStreamWaitEvent(st, e.ev_opt[chunk], 0));
  if (chunk + 1 == (int)e.ev_opt.size()) e.opt_pending = false;   // everything the optimizer wrote is now ordered before `st`
  return 0;
}

static int ensure_side_stream(Engine& e) {
  if (e.side) return 0;
  VQ_CUDA(cudaEventCreateWithFlags(&e.ev_gzero, cudaEventDisableTiming));
  VQ_CUDA(cudaStreamCreateWithFlags(&e.side, cudaStreamNonBlocking));
  VQ_CUDA(cudaEventCreateWithFlags(&e.ev_fork, cudaEventDisableTiming));
  VQ_CUDA(cudaEventCreateWithFlags(&e.ev_join, cudaEventDisableTiming));
  for (auto& ev : e.ev_layer) VQ_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  return 0;
}

// Two streams: `st` carries the dependency chain (dX GEMMs, attention and norm backward); every weight-gradient GEMM
// goes to the side stream `sd` right after the kernel that produced its dY operand (fork event). Nothing reads a dW
// before the optimizer, so the side stream fills the SMs the chain leaves idle — whole SMs for the decoder's small
// launches (M = B*T rows: 78-117 CTAs), wave tails for the encoder's. Write-after-read safety: every dY buffer the side
// stream reads comes from a ring 3 layers deep, and the main stream starts a layer only after the side stream has
// finished the layer two above it (ev_layer).
typedef void (*vq_stage_cb)(int stage, void* user);

static int backward(Engine& e, const float* w_rows, const float* gscale, int accumulate, int stage_begin, int stage_end, cudaStream_t st,
                    cudaStream_t comm = nullptr, vq_stage_cb cb = nullptr, void* cb_user = nullptr) {
  VQ_CHECK(e.fwd_valid, "engine: backward called without a preceding training forward");
  VQ_CHECK(e.G, "engine: gradient arena not bound");
  if (ensure_side_stream(e)) return 1;
  cudaStream_t sd = e.side;
  const vqacl_config& c = e.cfg;
  Workspace& w = e.w;
  const vqacl_batch& b = g_saved[&e].b;
  const int d = c.d_model, f = c.d_ff, H = c.n_heads, Ld = c.n_dec_layers, Le = c.n_enc_layers;
  const int B = b.B, L = b.L, N = b.N, T = b.T, S = L + N, S2 = S + 2;
  const int M = B * S, Md = B * T, M2 = B * S2;
  const int ldkv = Ld * 2 * d, V = c.vocab_size;
  constexpr int RING = Workspace::RING;
  const int n_stages = n_backward_stages(e);
  if (stage_end < 0 || stage_end > n_stages) stage_end = n_stages;
  VQ_CHECK(stage_begin >= 0 && stage_begin <= stage_end, "backward: bad stage range [%d, %d)", stage_begin, stage_end);
  auto on = [&](int s) { return s >= stage_begin && s < stage_end; };
  // side stream picks up everything the main stream has issued so far
  auto fork = [&]() -> int {
    VQ_CUDA(cudaEventRecord(e.ev_fork, st));
    VQ_CUDA(cudaStreamWaitEvent(sd, e.ev_fork, 0));
    return 0;
  };
  // end of a stage: the gradient range it finalised (backward_stage_range) is complete once BOTH streams reach this point
  auto stage_done = [&](int s) -> int {
    if (!cb) return 0;
    if ((int)e.ev_stage_main.size() < n_stages) {
      e.ev_stage_main.resize(n_stages, nullptr);
      e.ev_stage_side.resize(n_stages, nullptr);
      for (int i = 0; i < n_stages; ++i) {
        if (!e.ev_stage_main[i]) VQ_CUDA(cudaEventCreateWithFlags(&e.ev_stage_main[i], cudaEventDisableTiming));
        if (!e.ev_stage_side[i]) VQ_CUDA(cudaEventCreateWithFlags(&e.ev_stage_side[i], cudaEventDisableTiming));
      }
    }
    VQ_CUDA(cudaEventRecord(e.ev_stage_main[s], st));
    VQ_CUDA(cudaEventRecord(e.ev_stage_side[s], sd));
    VQ_CUDA(cudaStreamWaitEvent(comm, e.ev_stage_main[s], 0));
    VQ_CUDA(cudaStreamWaitEvent(comm, e.ev_stage_side[s], 0));
    cb(s, cb_user);   // the host enqueues the all-reduce(s) it planned for this stage on `comm`
    return 0;
  };
  int layer_no = 0;   // layers processed in this call (for the 2-layer lag)
  auto layer_begin = [&]() -> int {
    // the side stream must be done with the layer two above before its ring slots are rewritten
    if (layer_no >= 2) VQ_CUDA(cudaStreamWaitEvent(st, e.ev_layer[(layer_no - 2) & 3], 0));
    return 0;
  };
  auto layer_end = [&]() -> int {
    VQ_CUDA(cudaEventRecord(e.ev_layer[layer_no & 3], sd));
    ++layer_no;
    return 0;
  };
  if (on(0)) {
    if (!accumulate) {
      if (e.g_prezeroed) VQ_CUDA(cudaStreamWaitEvent(st, e.ev_gzero, 0));   // cleared during the decoder forward
      else VQ_CUDA(cudaMemsetAsync(e.G, 0, e.n_train * sizeof(float), st));
    }
    e.g_prezeroed = false;
    // ---- LM head + CE
    VQ_CHECK(w_rows, "backward: w_rows (dL/dloss_row) required");
    VQ_TRY(ce_bwd(w.logits, e.ldv, Md, V, b.labels, w.lse_ce, w_rows, gscale, st));
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(w.logits, e.ldv, w.yfin, d, e.G + e.o_shared, V, d, Md, sd));
    // dY_fin[Md, d] = dLogits[Md, V] * E[V, d]: few output tiles but a 32 200-deep contraction -> split-K into an fp32 buffer
    {
      const int tiles = ((Md + 127) / 128) * ((d + 255) / 256);
      int splits = num_sms() / (tiles > 0 ? tiles : 1);
      if (splits < 1) splits = 1;
      if (splits > 16) splits = 16;
      VQ_CUDA(cudaMemsetAsync(w.t_d768_f32, 0, (size_t)Md * d * sizeof(float), st));
      VQ_TRY(gemm_dx(w.logits, e.ldv, e.W + e.o_shared, V, d, w.t_d768_f32, d, Md, EPI_ATOMIC_F32, st, nullptr, 0, 1.f, splits));
    }
    e.gdb_i = 0;
    RmsBwdArgs r{};
    r.dn_f32 = w.t_d768_f32; r.dn_zero = 1; r.ld_dn = d; r.x = w.y[3 * Ld]; r.w = e.P + e.o_dec_final; r.g_in = nullptr; r.g_out = w.gd;
    r.gb_out = w.gdb_ring[e.gdb_i];
    r.dw = e.G + e.o_dec_final; r.M = Md; r.eps = c.eps; r.scale = 1.f / sqrtf((float)d); r.own = e.drop(SITE_DEC_FINAL);
    r.consumer = e.drop(site_dec(Ld - 1, 5)); r.consumer_cols = d;
    VQ_TRY(rmsnorm_bwd(r, st));
    VQ_TRY(stage_done(0));
  }
  for (int l = Ld - 1; l >= 0; --l) {
    if (!on(Ld - l)) continue;
    const DecLayer& P = e.dec[l];
    VQ_TRY(layer_begin());
    const int ri = l % RING;
    bf16* gdb_in = w.gdb_ring[e.gdb_i];
    bf16* gdb_1 = w.gdb_ring[(e.gdb_i + 1) % (3 * RING)];
    bf16* gdb_2 = w.gdb_ring[(e.gdb_i + 2) % (3 * RING)];
    bf16* gdb_out = w.gdb_ring[(e.gdb_i + 3) % (3 * RING)];
    e.gdb_i = (e.gdb_i + 3) % (3 * RING);
    // Weight gradients: with M = B*T rows of contraction each of the six dW GEMMs is a launch of 18-72 tiles whose pipeline fill
    // and drain outweigh its 25 k-blocks, and whose persistent CTAs (225 KB of shared memory) keep the chain's next kernel off
    // the SMs they hold. Grouped: the six problems are queued here and go out as ONE launch of 126 CTA-pair tiles on the side
    // stream at the end of the layer (their dY operands live in rings three layers deep).
    const bool grouped = g_dec_dw_grouped != 0 && gemm_pair_on();
    GemmGroupProblem dwq[6];
    int ndw = 0;
    auto dw = [&](const bf16* dY, int lddy, const bf16* X, int ldx, float* dWt, int n_out, int n_in) -> int {
      if (grouped) {
        dwq[ndw++] = GemmGroupProblem{dY, lddy, X, ldx, dWt, n_in, n_out, n_in};
        return 0;
      }
      VQ_TRY(fork());
      return gemm_dw(dY, lddy, X, ldx, dWt, n_out, n_in, Md, sd, g_dec_dw_sms);
    };
    // FFN
    VQ_TRY(dw(gdb_in, d, w.dh[l], f, e.G + P.wo, d, f));
    VQ_TRY(gemm_dx(gdb_in, d, e.W + P.wo, d, f, w.t_dh[ri], f, Md, EPI_RELUBWD_BF16, st, w.dhmask[l], (f + 31) / 32, e.drop(site_dec(l, 4)).inv_keep));
    VQ_TRY(dw(w.t_dh[ri], f, w.dn3[l], d, e.G + P.wi, f, d));
    // The deep contractions of the chain (dX of wi: K = d_ff, dX of qkv: K = 3 d) are split-K: with M = B*T rows there are only
    // 39-78 output tiles, and a CTA's operand stream is bound by its SM's ~120 GB/s L2 port (measured: 3.2 us + 0.27 us per 32 KB
    // k-block, tools/gemm_small_sweep.py) — three K slices per tile engage 126 SMs instead of 42. The slices meet in an fp32
    // buffer (red.global.add) that the RMSNorm backward reads — and clears for the next user — instead of a bf16 dX.
    const int dsplit = g_dec_dx_splits;
    if (dsplit > 1) VQ_TRY(gemm_dx(w.t_dh[ri], f, e.W + P.wi, f, d, w.t_d768_f32, d, Md, EPI_ATOMIC_F32, st, nullptr, 0, 1.f, dsplit));
    else VQ_TRY(gemm_dx(w.t_dh[ri], f, e.W + P.wi, f, d, w.t_d768, d, Md, EPI_BF16, st));
    RmsBwdArgs q{};
    q.dn = w.t_d768; q.ld_dn = d; q.x = w.y[3 * l + 2];
    if (dsplit > 1) { q.dn_f32 = w.t_d768_f32; q.dn_zero = 1; } q.w = e.P + P.ln2; q.g_in = w.gd; q.g_out = w.gd; q.gb_out = gdb_1;
    q.dw = e.G + P.ln2; q.M = Md; q.eps = c.eps; q.scale = 1.f; q.consumer = e.drop(site_dec(l, 3)); q.consumer_cols = d;
    VQ_TRY(rmsnorm_bwd(q, st));
    // cross attention
    VQ_TRY(dw(gdb_1, d, w.cao[l], d, e.G + P.co, d, d));
    VQ_TRY(gemm_dx(gdb_1, d, e.W + P.co, d, d, w.t_d768, d, Md, EPI_BF16, st));
    AttnArgs x{};
    x.q = w.cq[l]; x.ldq = d; x.k = w.kv_all + (size_t)l * 2 * d; x.v = x.k + d; x.ldk = x.ldv = ldkv;
    x.ldo = d; x.lse = w.lse_c[l]; x.B = B; x.H = H; x.Sq = T; x.Sk = S2; x.rel_mode = 0; x.keymask = w.cross_mask; x.causal = 0;
    Dropout dp = e.drop(site_dec(l, 2));
    x.drop_thr = dp.thr; x.drop_inv_keep = dp.inv_keep; x.seed = dp.seed; x.site = dp.site;
    x.o_saved = w.cao[l];
    x.dO = w.t_d768; x.dq = w.t_dcq[ri]; x.lddq = d; x.dk = w.dkv_all + (size_t)l * 2 * d; x.dv = x.dk + d; x.lddk = x.lddv = ldkv;
    VQ_TRY(attn_bwd(x, st));
    VQ_TRY(dw(w.t_dcq[ri], d, w.dn2[l], d, e.G + P.cq, d, d));
    VQ_TRY(gemm_dx(w.t_dcq[ri], d, e.W + P.cq, d, d, w.t_d768, d, Md, EPI_BF16, st));
    q.x = w.y[3 * l + 1]; q.w = e.P + P.ln1; q.dw = e.G + P.ln1; q.consumer = e.drop(site_dec(l, 1)); q.gb_out = gdb_2;
    q.dn_f32 = nullptr; q.dn_zero = 0;       // dX of cq (K = d) stays a bf16 single pass
    VQ_TRY(rmsnorm_bwd(q, st));
    // self attention
    VQ_TRY(dw(gdb_2, d, w.dao[l], d, e.G + P.o, d, d));
    VQ_TRY(gemm_dx(gdb_2, d, e.W + P.o, d, d, w.t_d768, d, Md, EPI_BF16, st));
    AttnArgs a{};
    a.q = w.dqkv[l]; a.k = w.dqkv[l] + d; a.v = w.dqkv[l] + 2 * d; a.ldq = a.ldk = a.ldv = 3 * d;
    a.ldo = d; a.lse = w.lse_s[l]; a.B = B; a.H = H; a.Sq = T; a.Sk = T;
    a.rel_table = e.P + e.o_dec_rel; a.rel_bucket = e.dec_bucket; a.rel_mode = 2; a.causal = 1;
    dp = e.drop(site_dec(l, 0));
    a.drop_thr = dp.thr; a.drop_inv_keep = dp.inv_keep; a.seed = dp.seed; a.site = dp.site;
    a.dO = w.t_d768; a.dq = w.t_dqkv[ri]; a.dk = w.t_dqkv[ri] + d; a.dv = w.t_dqkv[ri] + 2 * d; a.lddq = a.lddk = a.lddv = 3 * d;
    a.d_rel_table = e.G + e.o_dec_rel;
    VQ_TRY(attn_bwd(a, st));
    VQ_TRY(dw(w.t_dqkv[ri], 3 * d, w.dn1[l], d, e.G + P.qkv, 3 * d, d));
    if (dsplit > 1) VQ_TRY(gemm_dx(w.t_dqkv[ri], 3 * d, e.W + P.qkv, 3 * d, d, w.t_d768_f32, d, Md, EPI_ATOMIC_F32, st, nullptr, 0, 1.f, dsplit));
    else VQ_TRY(gemm_dx(w.t_dqkv[ri], 3 * d, e.W + P.qkv, 3 * d, d, w.t_d768, d, Md, EPI_BF16, st));
    if (dsplit > 1) { q.dn_f32 = w.t_d768_f32; q.dn_zero = 1; }
    q.x = w.y[3 * l]; q.w = e.P + P.ln0; q.dw = e.G + P.ln0; q.gb_out = gdb_out;
    q.consumer = l > 0 ? e.drop(site_dec(l - 1, 5)) : Dropout();
    VQ_TRY(rmsnorm_bwd(q, st));
    if (grouped) {
      VQ_TRY(fork());       // every dY of the layer has been produced
      VQ_TRY(gemm_bf16_grouped_mn(dwq, ndw, Md, EPI_ATOMIC_F32, 1.f, g_dec_dw_sms, sd));
    }
    VQ_TRY(layer_end());
    VQ_TRY(stage_done(Ld - l));
  }
  if (on(Ld + 1)) {
    // decoder token embedding (tied `shared`)
    VQ_TRY(embed_bwd(w.dec_ids, B, T, w.gd, T, 0, e.G + e.o_shared, e.drop(SITE_DEC_EMB), V, st));
    // cross-attention K/V projection of all layers: dW and the gradient flowing into the decoder memory
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(w.dkv_all, ldkv, w.mem, d, e.G + e.o_ckv, ldkv, d, M2, sd));
    VQ_TRY(gemm_dx(w.dkv_all, ldkv, e.W + e.o_ckv, ldkv, d, w.dmem, d, M2, EPI_BF16, st));
    // ---- encoder: final norm (rows S, S+1 of each memory slab are the detached prototypes -> dropped by the row map)
    e.geb_i = 0;
    RmsBwdArgs en{};
    en.dn = w.dmem; en.ld_dn = d; en.in_rpb = S; en.out_rpb = S2; en.x = w.x[2 * Le]; en.w = e.P + e.o_enc_final;
    en.g_in = nullptr; en.g_out = w.ge; en.gb_out = w.geb_ring[e.geb_i]; en.dw = e.G + e.o_enc_final; en.M = M; en.eps = c.eps; en.scale = 1.f;
    en.own = e.drop(SITE_ENC_FINAL); en.consumer = e.drop(site_enc(Le - 1, 3)); en.consumer_cols = d;
    if (e.mem_loss_valid && e.mem_loss_g) {
      // d loss_Q / d hidden[b,t,:] = 2 (mean_Q[b] - P_Q[label_b]) / (B * n_Q) for the n_Q tokens of the Q side, same for V
      const int nq = c.split_L < S ? c.split_L : S, nv = S - nq;
      en.bc_q = w.memdQ; en.bc_v = w.memdV; en.bc_g = e.mem_loss_g; en.bc_S = S; en.bc_split = nq;
      en.bc_cq = 2.f / ((float)B * (float)nq);
      en.bc_cv = nv > 0 ? 2.f / ((float)B * (float)nv) : 0.f;
    }
    VQ_TRY(rmsnorm_bwd(en, st));
    VQ_TRY(stage_done(Ld + 1));
  }
  for (int l = Le - 1; l >= 0; --l) {
    if (!on(Ld + 1 + Le - l)) continue;
    const EncLayer& P = e.enc[l];
    VQ_TRY(layer_begin());
    const int ri = l % RING;
    bf16* geb_in = w.geb_ring[e.geb_i];
    bf16* geb_1 = w.geb_ring[(e.geb_i + 1) % (2 * RING)];
    bf16* geb_out = w.geb_ring[(e.geb_i + 2) % (2 * RING)];
    e.geb_i = (e.geb_i + 2) % (2 * RING);
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(geb_in, d, w.h[l], f, e.G + P.wo, d, f, M, sd));
    VQ_TRY(gemm_dx(geb_in, d, e.W + P.wo, d, f, w.t_eh[ri], f, M, EPI_RELUBWD_BF16, st, w.hmask[l], (f + 31) / 32, e.drop(site_enc(l, 2)).inv_keep));
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(w.t_eh[ri], f, w.n2[l], d, e.G + P.wi, f, d, M, sd));
    VQ_TRY(gemm_dx(w.t_eh[ri], f, e.W + P.wi, f, d, w.t_e768, d, M, EPI_BF16, st));
    RmsBwdArgs q{};
    q.dn = w.t_e768; q.ld_dn = d; q.x = w.x[2 * l + 1]; q.w = e.P + P.ln1; q.g_in = w.ge; q.g_out = w.ge; q.gb_out = geb_1;
    q.dw = e.G + P.ln1; q.M = M; q.eps = c.eps; q.scale = 1.f; q.consumer = e.drop(site_enc(l, 1)); q.consumer_cols = d;
    VQ_TRY(rmsnorm_bwd(q, st));
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(geb_1, d, w.ao[l], d, e.G + P.o, d, d, M, sd));
    VQ_TRY(gemm_dx(geb_1, d, e.W + P.o, d, d, w.t_e768, d, M, EPI_BF16, st));
    AttnArgs a{};
    a.q = w.qkv[l]; a.k = w.qkv[l] + d; a.v = w.qkv[l] + 2 * d; a.ldq = a.ldk = a.ldv = 3 * d;
    a.ldo = d; a.lse = w.lse_e[l]; a.B = B; a.H = H; a.Sq = S; a.Sk = S;
    a.rel_table = e.P + e.o_enc_rel; a.rel_bucket = e.enc_bucket; a.rel_mode = 1; a.Lt = L; a.keymask = w.enc_mask; a.causal = 0;
    const Dropout dp = e.drop(site_enc(l, 0));
    a.drop_thr = dp.thr; a.drop_inv_keep = dp.inv_keep; a.seed = dp.seed; a.site = dp.site;
    a.dO = w.t_e768; a.dq = w.t_eqkv[ri]; a.dk = w.t_eqkv[ri] + d; a.dv = w.t_eqkv[ri] + 2 * d; a.lddq = a.lddk = a.lddv = 3 * d;
    a.d_rel_table = e.G + e.o_enc_rel;
    a.o_saved = w.ao[l];      // used by the multi-tile backward (S > 64): D = rowsum(dO * O)
    VQ_TRY(attn_bwd(a, st));
    VQ_TRY(fork());
    VQ_TRY(gemm_dw(w.t_eqkv[ri], 3 * d, w.n1[l], d, e.G + P.qkv, 3 * d, d, M, sd));
    VQ_TRY(gemm_dx(w.t_eqkv[ri], 3 * d, e.W + P.qkv, 3 * d, d, w.t_e768, d, M, EPI_BF16, st));
    q.x = w.x[2 * l]; q.w = e.P + P.ln0; q.dw = e.G + P.ln0; q.gb_out = geb_out;
    q.consumer = l > 0 ? e.drop(site_enc(l - 1, 3)) : Dropout();
    if (l == 0) q.gb_out = nullptr;
    VQ_TRY(rmsnorm_bwd(q, st));
    VQ_TRY(layer_end());
    VQ_TRY(stage_done(Ld + 1 + Le - l));
  }
  if (on(Ld + Le + 2)) {
    // ---- embeddings: text tokens (tied shared) and the VisualEmbedding
    VQ_TRY(embed_bwd(b.input_ids, B, L, w.ge, S, 0, e.G + e.o_shared, e.drop(SITE_ENC_EMB), V, st));
    VisArgs va{};
    va.featpre = w.featpre; va.boxes = b.boxes; va.bf = e.P + e.o_bf; va.wf = e.P + e.o_wf; va.Wp = e.P + e.o_Wp;
    va.bp = e.P + e.o_bp; va.wp = e.P + e.o_wp; va.img_emb = e.P + e.o_img; va.shared = e.P + e.o_shared;
    va.V = V; va.B = B; va.N = N; va.S = S; va.L = L; va.eps = c.eps; va.drop = e.drop(SITE_ENC_EMB);
    va.g = w.ge; va.dfeatpre = w.dfeatpre; va.dbf = e.G + e.o_bf; va.dwf = e.G + e.o_wf; va.dWp = e.G + e.o_Wp;
    va.dbp = e.G + e.o_bp; va.dwp = e.G + e.o_wp; va.dimg = e.G + e.o_img; va.dshared = e.G + e.o_shared;
    va.partials = w.vis_partials;
    VQ_TRY(vis_embed_bwd(va, st));
    VQ_TRY(gemm_dw(w.dfeatpre, d, b.vis_feats_bf16 ? reinterpret_cast<const bf16*>(b.vis_feats_bf16) : w.feats_bf16, c.feat_dim,
                   e.G + e.o_Wf, d, c.feat_dim, B * N, st));
    VQ_TRY(stage_done(Ld + Le + 2));
  }
  // join: the caller's stream owns every gradient written by this call
  VQ_CUDA(cudaEventRecord(e.ev_join, sd));
  VQ_CUDA(cudaStreamWaitEvent(st, e.ev_join, 0));
  // the last stage consumed the forward state (ce_bwd overwrote the logits with dLogits, the dY rings are spent): a second
  // backward on the same forward must fail loudly instead of accumulating garbage
  if (stage_end == n_stages) e.fwd_valid = false;
  return 0;
}

}  // namespace vq

// ===================================================================================================== C-ABI
using namespace vq;
#define ENG(p) (*reinterpret_cast<Engine*>(p))
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" int vqacl_engine_create(const vqacl_config* cfg, void** engine) {
  VQ_CHECK(cfg && engine, "engine_create: null argument");
  Engine* e = new Engine();
  e->cfg = *cfg;
  if (engine_build_layout(*e)) {
    delete e;
    return 1;
  }
  *engine = e;
  return 0;
}
extern "C" void vqacl_engine_destroy(void* engine) {
  if (!engine) return;
  {
    Engine& e = *reinterpret_cast<Engine*>(engine);
    if (e.opt_stream) {
      cudaStreamSynchronize(e.opt_stream);
      for (auto& ev : e.ev_opt) cudaEventDestroy(ev);
      cudaEventDestroy(e.ev_opt_fork);
      cudaStreamDestroy(e.opt_stream);
    }
    for (auto& ev : e.ev_stage_main) if (ev) cudaEventDestroy(ev);
    for (auto& ev : e.ev_stage_side) if (ev) cudaEventDestroy(ev);
    if (e.side) {
      cudaStreamSynchronize(e.side);
      cudaEventDestroy(e.ev_fork);
      cudaEventDestroy(e.ev_join);
      cudaEventDestroy(e.ev_gzero);
      for (auto& ev : e.ev_layer) cudaEventDestroy(ev);
      cudaStreamDestroy(e.side);
    }
  }
  if (reinterpret_cast<Engine*>(engine)->opt_scratch) cudaFree(reinterpret_cast<Engine*>(engine)->opt_scratch);
  g_saved.erase(reinterpret_cast<Engine*>(engine));
  delete reinterpret_cast<Engine*>(engine);
}
extern "C" int vqacl_param_count(void* engine) { return (int)ENG(engine).params.size(); }
extern "C" int vqacl_param_info(void* engine, int i, char* name, int name_cap, int64_t* offset, int* rows, int* cols, int* group) {
  Engine& e = ENG(engine);
  VQ_CHECK(i >= 0 && i < (int)e.params.size(), "param_info: index %d out of range", i);
  const ParamInfo& p = e.params[i];
  if (name && name_cap > 0) {
    strncpy(name, p.name.c_str(), name_cap - 1);
    name[name_cap - 1] = 0;
  }
  if (offset) *offset = (int64_t)p.off;
  if (rows) *rows = p.rows;
  if (cols) *cols = p.cols;
  if (group) *group = p.group;
  return 0;
}
extern "C" int64_t vqacl_arena_elems(void* engine, int64_t* n_decay, int64_t* n_train) {
  Engine& e = ENG(engine);
  if (n_decay) *n_decay = (int64_t)e.n_decay;
  if (n_train) *n_train = (int64_t)e.n_train;
  return (int64_t)e.n_total;
}
// first element of the tail region (see engine_build_layout): [0, tail) = GEMM-only matrices (sharded optimizer state with
// N > 1 GPUs), [tail, n_train) = parameters every rank keeps current in fp32
extern "C" int64_t vqacl_arena_tail(void* engine) { return (int64_t)ENG(engine).o_tail; }
extern "C" int vqacl_bind_arena(void* engine, float* params, float* grads, void* params_bf16) {
  Engine& e = ENG(engine);
  VQ_CHECK(params && params_bf16, "bind_arena: null arena");
  VQ_CHECK(((uintptr_t)params & 255) == 0 && ((uintptr_t)params_bf16 & 255) == 0 && ((uintptr_t)grads & 255) == 0,
           "bind_arena: arenas must be 256-byte aligned");
  e.P = params; e.G = grads; e.W = reinterpret_cast<bf16*>(params_bf16);
  if (!e.opt_scratch) {
    VQ_CUDA(cudaMalloc(&e.opt_scratch, (64 + Engine::OPT_PARTIALS) * sizeof(float)));
    VQ_CUDA(cudaMemset(e.opt_scratch, 0, (64 + Engine::OPT_PARTIALS) * sizeof(float)));
  }
  gemm_tmap_cache_clear();
  return 0;
}
extern "C" int vqacl_set_rel_buckets(void* engine, const int32_t* enc_b, const int32_t* dec_b) {
  Engine& e = ENG(engine);
  VQ_CHECK(enc_b && dec_b, "set_rel_buckets: null table");
  memcpy(e.enc_bucket_h, enc_b, 127 * sizeof(int32_t));   // HOST pointers: the maps travel in kernel parameters
  memcpy(e.dec_bucket_h, dec_b, 127 * sizeof(int32_t));
  e.enc_bucket = e.enc_bucket_h;
  e.dec_bucket = e.dec_bucket_h;
  return 0;
}
extern "C" int vqacl_refresh_bf16(void* engine, void* stream) {
  Engine& e = ENG(engine);
  VQ_CHECK(e.P && e.W, "refresh_bf16: arena not bound");
  return cast_f32_to_bf16(e.P, e.W, e.n_total, ST(stream));
}
extern "C" int64_t vqacl_workspace_bytes(void* engine, int B, int L, int N, int T) { return engine_carve(ENG(engine), nullptr, B, L, N, T); }
extern "C" int vqacl_bind_workspace(void* engine, void* ws, int64_t bytes, int B, int L, int N, int T) {
  Engine& e = ENG(engine);
  VQ_CHECK(ws && ((uintptr_t)ws & 255) == 0, "bind_workspace: workspace must be 256-byte aligned");
  const int64_t need = engine_carve(e, nullptr, B, L, N, T);
  VQ_CHECK(bytes >= need, "bind_workspace: %lld bytes given, %lld needed", (long long)bytes, (long long)need);
  engine_carve(e, reinterpret_cast<uint8_t*>(ws), B, L, N, T);
  gemm_tmap_cache_clear();
  return 0;
}
extern "C" int64_t vqacl_ws_offset(void* engine, const char* name) {
  Engine& e = ENG(engine);
  auto it = e.ws_names.find(name);
  return it == e.ws_names.end() ? -1 : it->second;
}

extern "C" int vqacl_forward_encoder(void* engine, const vqacl_batch* batch, const vqacl_proto_state* proto, uint32_t seed,
                                     int training, void* stream) {
  Engine& e = ENG(engine);
  (void)proto;
  if (check_batch(e, batch, training != 0)) return 1;
  e.seed = seed;
  e.training = training != 0;
  e.fwd_valid = false;
  return encoder_forward(e, batch, ST(stream));
}
extern "C" int vqacl_proto_sums(void* engine, const vqacl_batch* batch, void* stream) {
  Engine& e = ENG(engine);
  if (check_batch(e, batch, false)) return 1;
  VQ_CHECK(batch->cate_labels && batch->ques_labels, "proto_sums: needs cate_labels and ques_labels");
  VQ_TRY(proto_scatter_sum(e.w.meanQ, batch->ques_labels, batch->B, e.cfg.n_ques, e.w.curQ, e.w.cntQ, ST(stream)));
  VQ_TRY(proto_scatter_sum(e.w.meanV, batch->cate_labels, batch->B, e.cfg.n_cate, e.w.curV, e.w.cntV, ST(stream)));
  return 0;
}
extern "C" int vqacl_forward_decoder(void* engine, const vqacl_batch* batch, const vqacl_proto_state* proto, int sums_ready,
                                     int prezero_grads, void* stream) {
  Engine& e = ENG(engine);
  if (check_batch(e, batch, true)) return 1;
  VQ_CHECK(batch->labels || batch->decoder_input_ids, "forward_decoder: labels or decoder_input_ids required");
  e.prezero_request = prezero_grads != 0 && batch->labels;
  if (si_path(e, batch, proto, sums_ready != 0, ST(stream))) return 1;
  if (decoder_forward(e, batch, ST(stream))) return 1;
  g_saved[&e].b = *batch;
  e.fwd_valid = batch->labels != nullptr;      // logits-only calls (decoder_input_ids without labels) have no backward
  return 0;
}
extern "C" int vqacl_backward(void* engine, const float* w_rows, const float* gscale, int accumulate, int stage_begin, int stage_end,
                              void* stream) {
  return backward(ENG(engine), w_rows, gscale, accumulate, stage_begin, stage_end, ST(stream));
}
extern "C" int vqacl_backward_overlapped(void* engine, const float* w_rows, const float* gscale, int accumulate, void* comm_stream,
                                         void (*stage_cb)(int, void*), void* user, void* stream) {
  VQ_CHECK(comm_stream && stage_cb, "backward_overlapped: communication stream and stage callback required");
  return backward(ENG(engine), w_rows, gscale, accumulate, 0, -1, ST(stream), ST(comm_stream), stage_cb, user);
}
// d(total loss) / d(loss_memory_Q, loss_memory_V) for the next backward (device float[2]; null = the memory losses do not
// take part in the objective). Only meaningful after a forward with vqacl_proto_state.memory_loss set.
extern "C" int vqacl_set_memory_loss_grads(void* engine, const float* g2) {
  ENG(engine).mem_loss_g = g2;
  return 0;
}
extern "C" int vqacl_backward_stages(void* engine) { return n_backward_stages(ENG(engine)); }
extern "C" int vqacl_backward_stage_range(void* engine, int stage, int64_t* begin, int64_t* end) {
  Engine& e = ENG(engine);
  VQ_CHECK(stage >= 0 && stage < n_backward_stages(e) && begin && end, "backward_stage_range: bad arguments");
  backward_stage_range(e, stage, begin, end);
  return 0;
}
extern "C" int vqacl_loss_tail(const float* loss_rows, const int64_t* labels, const float* scores, int B, int T, float* loss_out,
                               float* w_rows, void* stream) {
  return loss_tail(loss_rows, labels, scores, B, T, loss_out, w_rows, ST(stream));
}
static int g_opt_blocks_per_sm = [] { const char* ev = getenv("VQACL_OPT_BLOCKS_PER_SM"); return ev ? atoi(ev) : 2; }();
static AdamArgs adam_range(const Engine& e, float* m, float* v, size_t b, size_t en, float lr, float beta1, float beta2, float eps,
                           float weight_decay, int step, float max_norm) {
  AdamArgs a{};
  a.p = e.P + b; a.g = e.G + b; a.m = m + b; a.v = v + b; a.p_bf16 = e.W + b; a.n = en - b;
  a.n_decay = e.n_decay > b ? (e.n_decay - b < a.n ? e.n_decay - b : a.n) : 0;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay; a.step = step;
  a.sumsq = e.sumsq(); a.max_norm = max_norm;
  return a;
}

extern "C" int vqacl_clip_adamw(void* engine, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                                float weight_decay, int step, float max_grad_norm, float* grad_norm_out, int overlap, void* stream) {
  Engine& e = ENG(engine);
  cudaStream_t st = ST(stream);
  VQ_CHECK(e.P && e.G && e.W && e.ws_base, "clip_adamw: arena / workspace not bound");
  if (e.opt_pending) {   // a previous overlapped step that no forward consumed: order it before this one
    VQ_CUDA(cudaStreamWaitEvent(st, e.ev_opt.back(), 0));
    e.opt_pending = false;
  }
  VQ_TRY(grad_sumsq(e.G, e.n_train, e.sumsq_partials(), e.sumsq(), st));
  if (grad_norm_out) VQ_CUDA(cudaMemcpyAsync(grad_norm_out, e.sumsq(), sizeof(float), cudaMemcpyDeviceToDevice, st));
  if (!overlap) {
    VQ_TRY(adamw_hf(adam_range(e, exp_avg, exp_avg_sq, 0, e.n_train, lr, beta1, beta2, eps, weight_decay, step, max_grad_norm), st));
    return 0;
  }
  // ---- overlapped: the update is HBM-bound (30 B/param), the next forward's encoder GEMMs are tensor-bound. Update the arena
  //      in the order the forward reads it, on a separate stream; forward_encoder/decoder wait per chunk (wait_params).
  const int Le = e.cfg.n_enc_layers;
  if (!e.opt_stream) {
    VQ_CUDA(cudaStreamCreateWithFlags(&e.opt_stream, cudaStreamNonBlocking));
    VQ_CUDA(cudaEventCreateWithFlags(&e.ev_opt_fork, cudaEventDisableTiming));
    e.ev_opt.resize(Le + 2);
    for (auto& ev : e.ev_opt) VQ_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
  }
  VQ_CUDA(cudaEventRecord(e.ev_opt_fork, st));
  VQ_CUDA(cudaStreamWaitEvent(e.opt_stream, e.ev_opt_fork, 0));
  // 2 CTAs of 256 threads per SM: an AdamW grid that floods every SM's thread slots (8 CTAs = 2048 threads) keeps the forward's
  // persistent GEMM CTAs (384 threads, all of the SM's shared memory) from becoming resident until it drains; two CTAs fit
  // beside one and still hold ~64 KB of loads in flight per SM
  const int opt_blocks = g_opt_blocks_per_sm * num_sms();
  auto chunk = [&](int k, size_t b, size_t en) -> int {
    if (en > b) {
      AdamArgs aa = adam_range(e, exp_avg, exp_avg_sq, b, en, lr, beta1, beta2, eps, weight_decay, step, max_grad_norm);
      aa.max_blocks = opt_blocks;
      VQ_TRY(adamw_hf(aa, e.opt_stream));
    }
    VQ_CUDA(cudaEventRecord(e.ev_opt[k], e.opt_stream));
    return 0;
  };
  VQ_TRY(chunk(0, e.o_Wf, e.n_train));     // visual projection + tail (embeddings, every norm weight, biases): read first
  for (int l = 0; l < Le; ++l) VQ_TRY(chunk(1 + l, e.enc[l].qkv, l + 1 < Le ? e.enc[l + 1].qkv : e.o_Wf));
  VQ_TRY(chunk(1 + Le, 0, Le > 0 ? e.enc[0].qkv : e.o_Wf));
  e.opt_pending = true;
  return 0;
}
// ---- sharded optimizer (N > 1 GPUs): each rank owns the slices of the arena its bucketed reduce-scatter left it with
extern "C" int vqacl_grad_sumsq_ranges(void* engine, const int64_t* begin, const int64_t* end, int n_ranges, float* out, void* stream) {
  Engine& e = ENG(engine);
  VQ_CHECK(e.G && e.opt_scratch && out, "grad_sumsq_ranges: arena not bound");
  return grad_sumsq_ranges(e.G, begin, end, n_ranges, e.sumsq_partials(), Engine::OPT_PARTIALS, out, ST(stream));
}
// AdamW (+ clip by *sumsq, + bf16 refresh) over arena elements [begin, end); m / v point at the moments of element `begin`
extern "C" int vqacl_adamw_range(void* engine, float* m, float* v, int64_t begin, int64_t end, float lr, float beta1, float beta2, float eps,
                                 float weight_decay, int step, const float* sumsq, float max_grad_norm, void* stream) {
  Engine& e = ENG(engine);
  VQ_CHECK(e.P && e.G && e.W, "adamw_range: arena not bound");
  VQ_CHECK(begin >= 0 && begin <= end && (size_t)end <= e.n_train, "adamw_range: bad range [%lld, %lld)", (long long)begin, (long long)end);
  if (end == begin) return 0;
  AdamArgs a = adam_range(e, m - begin, v - begin, (size_t)begin, (size_t)end, lr, beta1, beta2, eps, weight_decay, step, max_grad_norm);
  a.sumsq = sumsq;
  return adamw_hf(a, ST(stream));
}

// order everything a pending overlapped optimizer step wrote before `stream` (state_dict(), evaluation, user code)
// Sharded optimizer (N > 1): events of the HOST's communication stream after which parameter chunk k (0: visual projection +
// tail, 1..Le: encoder layer k-1, Le+1: decoder + cross-KV) holds every rank's refreshed bf16 weights; the next
// forward_encoder / forward_decoder / generate waits chunk by chunk. The events must stay alive until that forward was issued.
extern "C" int vqacl_set_param_events(void* engine, void* const* events, int n) {
  Engine& e = ENG(engine);
  VQ_CHECK(n == 0 || n == e.cfg.n_enc_layers + 2, "set_param_events: %d events given, %d chunks", n, e.cfg.n_enc_layers + 2);
  e.ext_ev.assign(n, nullptr);
  for (int i = 0; i < n; ++i) e.ext_ev[i] = reinterpret_cast<cudaEvent_t>(events[i]);
  e.ext_pending = n > 0;
  return 0;
}
extern "C" int vqacl_param_sync(void* engine, void* stream) {
  Engine& e = ENG(engine);
  if (e.ext_pending) {
    for (cudaEvent_t ev : e.ext_ev)
      if (ev) VQ_CUDA(cudaStreamWaitEvent(ST(stream), ev, 0));
    e.ext_pending = false;
  }
  if (e.opt_pending) {
    VQ_CUDA(cudaStreamWaitEvent(ST(stream), e.ev_opt.back(), 0));
    e.opt_pending = false;
  }
  return 0;
}

// Device-side error flags raised by kernels that cannot fail synchronously (bit 0: token id outside [0, vocab) in an embedding
// gather — torch raises IndexError there). Synchronises `stream`, returns the flags and clears them.
extern "C" int vqacl_device_errors(void* engine, int* flags_out, void* stream) {
  Engine& e = ENG(engine);
  VQ_CHECK(flags_out, "device_errors: null output");
  *flags_out = 0;
  if (!e.opt_scratch) return 0;
  VQ_CUDA(cudaMemcpyAsync(flags_out, e.err_flags(), sizeof(int), cudaMemcpyDeviceToHost, ST(stream)));
  VQ_CUDA(cudaStreamSynchronize(ST(stream)));
  if (*flags_out) VQ_CUDA(cudaMemsetAsync(e.err_flags(), 0, sizeof(int), ST(stream)));
  return 0;
}

// ---- individual operators
extern "C" int vqacl_rmsnorm_fwd(const float* x, const float* w, void* y_bf16, float* y_f32, int M, float eps, float scale, void* stream) {
  RmsFwdArgs r{};
  r.x = x; r.w = w; r.y_bf16 = reinterpret_cast<bf16*>(y_bf16); r.ld_bf16 = DM; r.y_f32 = y_f32; r.ld_f32 = DM; r.M = M; r.eps = eps; r.scale = scale;
  return rmsnorm_fwd(r, ST(stream));
}
extern "C" int vqacl_rmsnorm_bwd(const void* dn_bf16, const float* x, const float* w, const float* g_in, float* g_out, void* gb_out,
                                 float* dw, int M, float eps, float scale, void* stream) {
  RmsBwdArgs r{};
  r.dn = reinterpret_cast<const bf16*>(dn_bf16); r.ld_dn = DM; r.x = x; r.w = w; r.g_in = g_in; r.g_out = g_out;
  r.gb_out = reinterpret_cast<bf16*>(gb_out); r.dw = dw; r.M = M; r.eps = eps; r.scale = scale; r.consumer_cols = DM;
  return rmsnorm_bwd(r, ST(stream));
}
static AttnArgs make_attn(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, int ldo, float* lse, int B, int H,
                          int Sq, int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt,
                          const float* keymask, int causal) {
  AttnArgs a{};
  a.q = reinterpret_cast<const bf16*>(q); a.k = reinterpret_cast<const bf16*>(k); a.v = reinterpret_cast<const bf16*>(v);
  a.ldq = ldq; a.ldk = ldk; a.ldv = ldv; a.ldo = ldo; a.lse = lse; a.B = B; a.H = H; a.Sq = Sq; a.Sk = Sk;
  a.rel_table = rel_table; a.rel_bucket = rel_bucket; a.rel_mode = rel_mode; a.Lt = Lt; a.keymask = keymask; a.causal = causal;
  return a;
}
extern "C" int vqacl_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, void* o, int ldo, float* lse,
                                   int B, int H, int Sq, int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode,
                                   int Lt, const float* keymask, int causal, void* stream) {
  AttnArgs a = make_attn(q, k, v, ldq, ldk, ldv, ldo, lse, B, H, Sq, Sk, rel_table, rel_bucket, rel_mode, Lt, keymask, causal);
  a.o = reinterpret_cast<bf16*>(o);
  return attn_fwd(a, ST(stream));
}
extern "C" int vqacl_attention_bwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, const void* dO, int ldo,
                                   const float* lse, void* dq, void* dk, void* dv, int lddq, int lddk, int lddv, int B, int H, int Sq,
                                   int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt,
                                   const float* keymask, int causal, float* d_rel_table, const void* o_saved, void* stream) {
  AttnArgs a = make_attn(q, k, v, ldq, ldk, ldv, ldo, const_cast<float*>(lse), B, H, Sq, Sk, rel_table, rel_bucket, rel_mode, Lt,
                         keymask, causal);
  a.dO = reinterpret_cast<const bf16*>(dO);
  a.dq = reinterpret_cast<bf16*>(dq); a.dk = reinterpret_cast<bf16*>(dk); a.dv = reinterpret_cast<bf16*>(dv);
  a.lddq = lddq; a.lddk = lddk; a.lddv = lddv; a.d_rel_table = d_rel_table;
  a.o_saved = reinterpret_cast<const bf16*>(o_saved);
  return attn_bwd(a, ST(stream));
}
extern "C" int vqacl_attention_fwd_ex(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, void* o, int ldo,
                                      float* lse, int B, int H, int Sq, int Sk, const float* rel_table, const int32_t* rel_bucket,
                                      int rel_mode, int Lt, const float* keymask, int causal, uint32_t drop_thr16, float inv_keep,
                                      uint32_t drop_key, int64_t q_bstride, int64_t k_bstride, int64_t v_bstride, int64_t o_bstride,
                                      int q_off, void* stream) {
  AttnArgs a = make_attn(q, k, v, ldq, ldk, ldv, ldo, lse, B, H, Sq, Sk, rel_table, rel_bucket, rel_mode, Lt, keymask, causal);
  a.o = reinterpret_cast<bf16*>(o);
  a.drop_thr = drop_thr16; a.drop_inv_keep = inv_keep; a.seed = drop_key;
  a.q_bstride = q_bstride; a.k_bstride = k_bstride; a.v_bstride = v_bstride; a.o_bstride = o_bstride; a.q_off = q_off;
  return attn_fwd(a, ST(stream));
}
extern "C" int vqacl_attention_bwd_ex(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, const void* dO, int ldo,
                                      const float* lse, void* dq, void* dk, void* dv, int lddq, int lddk, int lddv, int B, int H, int Sq,
                                      int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt,
                                      const float* keymask, int causal, float* d_rel_table, const void* o_saved, uint32_t drop_thr16,
                                      float inv_keep, uint32_t drop_key, void* stream) {
  AttnArgs a = make_attn(q, k, v, ldq, ldk, ldv, ldo, const_cast<float*>(lse), B, H, Sq, Sk, rel_table, rel_bucket, rel_mode, Lt,
                         keymask, causal);
  a.dO = reinterpret_cast<const bf16*>(dO);
  a.dq = reinterpret_cast<bf16*>(dq); a.dk = reinterpret_cast<bf16*>(dk); a.dv = reinterpret_cast<bf16*>(dv);
  a.lddq = lddq; a.lddk = lddk; a.lddv = lddv; a.d_rel_table = d_rel_table;
  a.o_saved = reinterpret_cast<const bf16*>(o_saved);
  a.drop_thr = drop_thr16; a.drop_inv_keep = inv_keep; a.seed = drop_key;
  return attn_bwd(a, ST(stream));
}
extern "C" int vqacl_proto_means(const float* h, int B, int S, int split, float* meanQ, float* meanV, void* stream) {
  return proto_means(h, B, S, split, meanQ, meanV, ST(stream));
}
extern "C" int vqacl_proto_scatter_mean(const float* mean, const float* labels, int B, int C, float* proto, float* cnt, void* stream) {
  return proto_scatter_mean(mean, labels, B, C, proto, cnt, ST(stream));
}
extern "C" int vqacl_proto_update(const float* curQ, const float* curV, const float* cntQ, const float* cntV, float* Qproto,
                                  float* Vproto, float* numQ, float* numV, int CQ, int CV, int task_id, int first_step_of_task,
                                  int has_mem, float alpha, float beta, void* stream) {
  ProtoUpdateArgs u{};
  u.curQ = curQ; u.curV = curV; u.cntQ = cntQ; u.cntV = cntV; u.Qproto = Qproto; u.Vproto = Vproto; u.numQ = numQ; u.numV = numV;
  u.CQ = CQ; u.CV = CV; u.task_id = task_id; u.first_step_of_task = first_step_of_task; u.has_mem = has_mem; u.alpha = alpha; u.beta = beta;
  return proto_update(u, ST(stream));
}
extern "C" int vqacl_proto_retrieve(const float* P, int C, const float* x, int B, void* out_bf16, int out_pitch_rows, int out_row,
                                    int64_t* idx, float* out_f32, float* scratch, void* stream) {
  return proto_retrieve(P, C, x, B, reinterpret_cast<bf16*>(out_bf16), out_pitch_rows, out_row, idx, out_f32, scratch, ST(stream));
}
extern "C" int vqacl_ce_fwd(const void* logits, int ld, int M, int V, const int64_t* labels, float* lse, float* loss, void* stream) {
  return ce_fwd(reinterpret_cast<const bf16*>(logits), ld, M, V, labels, lse, loss, ST(stream));
}
extern "C" int vqacl_ce_bwd(void* logits, int ld, int M, int V, const int64_t* labels, const float* lse, const float* w, void* stream) {
  return ce_bwd(reinterpret_cast<bf16*>(logits), ld, M, V, labels, lse, w, nullptr, ST(stream));
}
extern "C" int vqacl_visual_embed_fwd(const float* featpre, const float* boxes, const float* bf, const float* wf, const float* Wp,
                                      const float* bp, const float* wp, const float* img_emb, const float* shared, int V, int B,
                                      int N, int S, int L, float eps, float* x, void* stream) {
  VisArgs va{};
  va.featpre = featpre; va.boxes = boxes; va.bf = bf; va.wf = wf; va.Wp = Wp; va.bp = bp; va.wp = wp; va.img_emb = img_emb;
  va.shared = shared; va.V = V; va.B = B; va.N = N; va.S = S; va.L = L; va.eps = eps; va.x = x;
  return vis_embed_fwd(va, ST(stream));
}
extern "C" int vqacl_collate_device(const float* boxes_px, const float* img_wh, int B, int N, float* boxes_out, const int64_t* cate_ids,
                                    int n_cate, float* cate_onehot, const int64_t* ques_ids, int n_ques, float* ques_onehot, void* stream) {
  VQ_CHECK(boxes_px && img_wh && boxes_out, "collate_device: null box buffers");
  VQ_CHECK((!cate_ids || cate_onehot) && (!ques_ids || ques_onehot), "collate_device: ids without an output buffer");
  return collate_device(boxes_px, img_wh, B, N, boxes_out, cate_ids, n_cate, cate_onehot, ques_ids, n_ques, ques_onehot, ST(stream));
}
extern "C" int vqacl_adamw_hf(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n, int64_t n_decay, float lr,
                              float beta1, float beta2, float eps, float weight_decay, int step, const float* sumsq, float max_norm,
                              void* stream) {
  AdamArgs a{};
  a.p = p; a.g = g; a.m = m; a.v = v; a.p_bf16 = reinterpret_cast<bf16*>(p_bf16); a.n = (size_t)n; a.n_decay = (size_t)n_decay;
  a.lr = lr; a.beta1 = beta1; a.beta2 = beta2; a.eps = eps; a.weight_decay = weight_decay; a.step = step; a.sumsq = sumsq; a.max_norm = max_norm;
  return adamw_hf(a, ST(stream));
}
extern "C" int vqacl_grad_sumsq(const float* g, int64_t n, float* partials, float* out, void* stream) {
  return grad_sumsq(g, (size_t)n, partials, out, ST(stream));
}
