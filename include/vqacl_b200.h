/* vqacl_b200 — C-ABI of the B200-native VQACL hot path (VL-T5 train step + SI prototype bank + greedy decode).
 *
 * The reference (zhangxi1997/VQACL) is pure Python: its "FFI" for this path is the Python model-class API
 *   VLT5VQA.train_step / test_step      VL-T5/src/vqa_model.py:18-121
 *   VLT5.forward / prototype methods    VL-T5/src/modeling_t5_our.py:434-713
 *   Trainer.train_step tail             VL-T5/src/vqacl.py:429-509
 * which `vqacl_b200/` mirrors in Python on top of the entry points below (ctypes; see INTEGRATION.md).
 * Conventions: every function returns 0 on success; on failure it returns non-zero and vqacl_last_error() holds the
 * message (the Python host raises). All data pointers are DEVICE pointers unless stated; `stream` is a cudaStream_t.
 * No torch types cross this boundary. There is no CPU fallback.
 */
#ifndef VQACL_B200_H
#define VQACL_B200_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* vqacl_last_error(void);

/* ---- model configuration (trainer_base.py:57-89 + t5-base hyper-parameters) ---- */
typedef struct vqacl_config {
  int vocab_size;       /* 32200 (tokenization.py:58-60, vqacl.py:98-99) */
  int d_model;          /* 768 (kernels are specialised for it) */
  int d_kv;             /* 64 */
  int n_heads;          /* 12 */
  int d_ff;             /* 3072 */
  int n_enc_layers;     /* 12 */
  int n_dec_layers;     /* 12 */
  int n_buckets;        /* 32 */
  int feat_dim;         /* 2048 */
  int n_images;         /* 2 */
  int n_ques;           /* 10 question-type prototypes */
  int n_cate;           /* 80 object-category prototypes */
  int split_L;          /* 20: VLT5.L, the hard-coded Q/V split (modeling_t5_our.py:381) */
  int pad_id, eos_id, start_id; /* 0, 1, 0 */
  float eps;            /* 1e-6 */
  float dropout;        /* dropout_rate (param.py --dropout) */
} vqacl_config;

/* one step's inputs: what VLT5VQA.train_step moves to the device (vqa_model.py:20-27) */
typedef struct vqacl_batch {
  int B, L, N, T;              /* batch, text width, boxes per image, target width */
  const float* vis_feats;      /* [B,N,feat_dim] fp32 */
  const float* boxes;          /* [B,N,4] fp32 */
  const int64_t* input_ids;    /* [B,L] */
  const int64_t* labels;       /* [B,T], -100 = ignore (train only) */
  const float* cate_labels;    /* [B,n_cate] one-hot fp32 (train only) */
  const float* ques_labels;    /* [B,n_ques] one-hot fp32 (train only) */
  const int64_t* decoder_input_ids; /* optional [B,T]: explicit decoder inputs (VLT5.forward(decoder_input_ids=...),
                                  modeling_t5_our.py:617-629) instead of shift_right(labels); labels may then be NULL: the call
                                  produces logits only (no loss, no backward) */
  const void* vis_feats_bf16;  /* optional [B,N,feat_dim] bf16: RoI features already in the GEMM operand format (packed feature
                                  shards, vqacl_b200/pipeline.py). When set, vis_feats may be NULL and the fp32->bf16 cast is
                                  skipped; results are bit-identical to passing the fp32 values they were rounded from. */
} vqacl_batch;

/* SI prototype bank state (the reference keeps these as Python attributes of VLT5, modeling_t5_our.py:391-396) */
typedef struct vqacl_proto_state {
  float* Q_prototype;          /* [n_ques, d] persistent bank (== Q_task_mem_proto[t] storage for t > 0) */
  float* V_prototype;          /* [n_cate, d] */
  float* Q_num;                /* [n_ques] running counts */
  float* V_num;                /* [n_cate] */
  int proto_update;            /* kwargs['proto_update'] (train) */
  int task_id;                 /* current_task_id */
  int first_step_of_task;      /* current_task_id not in Q_task_cur_proto */
  int has_mem;                 /* current_task_id in Q_task_mem_proto */
  float alpha, beta;           /* --proto_alpha / --proto_beta */
  int memory_loss;             /* kwargs['memory'] (modeling_t5_our.py:590-592): also compute the prototype pull losses of
                                  nextqa/modeling_t5_nextqa.py:544-555 against the banks as they stand BEFORE this step's update;
                                  results in the workspace region "loss_memory" (float[2]: Q, V) */
} vqacl_proto_state;

/* ---- engine lifecycle ---- */
int vqacl_engine_create(const vqacl_config* cfg, void** engine);
void vqacl_engine_destroy(void* engine);
/* parameter arena: one flat fp32 buffer; the reference's state_dict tensors are views at these offsets */
int vqacl_param_count(void* engine);
int vqacl_param_info(void* engine, int i, char* name, int name_cap, int64_t* offset, int* rows, int* cols, int* group);
int64_t vqacl_arena_elems(void* engine, int64_t* n_decay, int64_t* n_train);
int vqacl_bind_arena(void* engine, float* params, float* grads, void* params_bf16);
/* relative-position bucket maps, HOST int32[127] each: bucket of (key - query + 63); computed by the host with the HF formula
 * (T5Attention._relative_position_bucket); they are copied and passed to the attention kernels as kernel parameters */
int vqacl_set_rel_buckets(void* engine, const int32_t* enc_bidirectional, const int32_t* dec_unidirectional);
int vqacl_refresh_bf16(void* engine, void* stream);                 /* params fp32 -> bf16 GEMM copies */
/* activation workspace: allocated by the host (torch caching allocator), carved by the engine */
int64_t vqacl_workspace_bytes(void* engine, int B, int L, int N, int T);
int vqacl_bind_workspace(void* engine, void* ws, int64_t bytes, int B, int L, int N, int T);
int64_t vqacl_ws_offset(void* engine, const char* name);            /* byte offset of a named output, -1 if unknown */

/* ---- hot path: VLT5.forward with labels (modeling_t5_our.py:514-713), split where the multi-GPU SI exchange sits ---- */
int vqacl_forward_encoder(void* engine, const vqacl_batch* batch, const vqacl_proto_state* proto, uint32_t seed, int training, void* stream);
/* multi-GPU SI exchange (SURVEY.md §8e): after forward_encoder, write the UN-divided per-class feature sums and counts of
 * this rank's batch into the workspace regions "curQ" [n_ques,d], "curV" [n_cate,d], "cntQ", "cntV"; the host all-reduces
 * (sum) them and passes sums_ready = 1 to forward_decoder, which then divides instead of recomputing. */
int vqacl_proto_sums(void* engine, const vqacl_batch* batch, void* stream);
/* prezero_grads != 0: the caller promises that the coming backward does NOT accumulate into existing gradients; the arena is
 * then cleared on a side stream during the decoder forward instead of at the start of backward. */
int vqacl_forward_decoder(void* engine, const vqacl_batch* batch, const vqacl_proto_state* proto, int sums_ready,
                          int prezero_grads, void* stream);
/* backward of sum_r w[r] * loss_row[r] (loss.backward(), vqacl.py:461); fills the gradient arena (zeroed in stage 0 unless
 * accumulate != 0). Runs stages [stage_begin, stage_end) (stage_end < 0: to the end) so that the host can overlap the NCCL
 * all-reduce of a finished arena range (vqacl_backward_stage_range) with the remaining stages. */
int vqacl_backward(void* engine, const float* w_rows, const float* gscale /* optional device scalar: upstream d(loss) */,
                   int accumulate, int stage_begin, int stage_end, void* stream);
/* whole backward in ONE call for N > 1 GPUs: after each stage the engine makes `comm_stream` wait for that stage on both of
 * its streams and calls stage_cb(stage, user); the host enqueues the all-reduce of vqacl_backward_stage_range(stage) (or of
 * a merged bucket) on comm_stream from inside the callback and joins comm_stream with `stream` afterwards. */
int vqacl_backward_overlapped(void* engine, const float* w_rows, const float* gscale, int accumulate, void* comm_stream,
                              void (*stage_cb)(int stage, void* user), void* user, void* stream);
/* weights of the two memory losses in the objective for the next backward: device float[2] = d loss / d (loss_memory_Q,
 * loss_memory_V), i.e. (lambda_Q, lambda_V) * upstream gradient (vqacl.py:448-450); NULL = not part of the objective */
int vqacl_set_memory_loss_grads(void* engine, const float* g2);
int vqacl_backward_stages(void* engine);
int vqacl_backward_stage_range(void* engine, int stage, int64_t* begin, int64_t* end);
/* fused loss tail of VLT5VQA.train_step (vqa_model.py:46-54) */
int vqacl_loss_tail(const float* loss_rows, const int64_t* labels, const float* scores, int B, int T, float* loss_out, float* w_rows, void* stream);
/* clip_grad_norm_ + HF AdamW + bf16 refresh (vqacl.py:475-482, trainer_base.py:130-198) */
int vqacl_clip_adamw(void* engine, float* exp_avg, float* exp_avg_sq, float lr, float beta1, float beta2, float eps,
                     float weight_decay, int step, float max_grad_norm, float* grad_norm_out, int overlap, void* stream);
/* overlap != 0: the (HBM-bound) update runs on an internal stream in the order the next forward reads the parameters and
 * vqacl_forward_encoder/decoder/generate wait chunk by chunk; any OTHER consumer of the parameters must call
 * vqacl_param_sync(engine, its_stream) first. */
int vqacl_param_sync(void* engine, void* stream);
/* Sharded step tail for N > 1 GPUs (what the reference's DDP + per-rank AdamW would do, vqacl.py:125-129,466-487, with the
 * optimizer state partitioned): after a bucketed reduce-scatter each rank owns some slices of the gradient arena.
 * vqacl_grad_sumsq_ranges: *out (device fp32) = sum of squares over the given arena ranges (host int64 arrays);
 * vqacl_adamw_range: clip (by *sumsq, the all-reduced global value) + HF AdamW + bf16 refresh over arena elements
 * [begin, end); m / v point at the moment buffers of element `begin`. */
int64_t vqacl_arena_tail(void* engine);   /* arena layout: [0, tail) GEMM-only matrices (sharded), [tail, n_train) replicated */
int vqacl_set_param_events(void* engine, void* const* events, int n);   /* cudaEvent_t per parameter chunk; see engine.cu */
int vqacl_grad_sumsq_ranges(void* engine, const int64_t* begin, const int64_t* end, int n_ranges, float* out, void* stream);
int vqacl_adamw_range(void* engine, float* m, float* v, int64_t begin, int64_t end, float lr, float beta1, float beta2, float eps,
                      float weight_decay, int step, const float* sumsq, float max_grad_norm, void* stream);
/* Errors kernels cannot raise synchronously (bit 0: a token id outside [0, vocab) reached an embedding gather — torch
 * raises IndexError at modeling_t5_our.py:196). Synchronises `stream`, returns and clears the flags (HOST int). */
int vqacl_device_errors(void* engine, int* flags_out, void* stream);
/* greedy generation (vqa_model.py:112-116; HF 4.2.1 generate/greedy_search with max_length 20, SURVEY.md H12):
 * out_tokens [B, max_len] int64 (column 0 = start token, finished rows emit pad); *out_len = columns produced.
 * The LM head runs with the argmax fused into its epilogue (fp32 accumulators; no [B, V] logits); the all-rows-finished test
 * HF does after every token synchronises the stream once per 4 tokens here (finished rows emit pad, the result is identical). */
int64_t vqacl_generate_workspace_bytes(void* engine, int B, int L, int N, int max_len);
int vqacl_generate(void* engine, const vqacl_batch* batch, const vqacl_proto_state* proto, int max_len, int64_t* out_tokens,
                   void* workspace, int64_t workspace_bytes, int* out_len, void* stream);
/* SMs the persistent GEMM kernels may occupy (0 = all): lowered by the host while an NCCL all-reduce must make progress
 * next to backward (the GEMM CTAs otherwise fill every SM's shared memory and starve the collective's CTAs) */
int vqacl_set_gemm_sm_limit(int n_sms);
/* dynamic (atomic-counter) tile schedule of the CTA-pair GEMM instead of the static round robin: a pair that becomes
 * resident late (its SMs were held by a collective or by another stream's kernel) finds the work list drained */
int vqacl_set_gemm_dynamic_schedule(int on);
/* number of kernels this library has launched so far in this process (bench.py's gpu_launches) */
long long vqacl_launch_count(void);

/* ---- individual operators (unit-test / building-block surface); `rel_bucket` is a HOST int32[127] table ----
 * Each entry replaces library calls the reference reaches through PyTorch / transformers 4.2.1:                              */

/* nn.Linear forward / input-gradient / weight-gradient (every q,k,v,o,wi,wo, feat_embedding.0 and the tied lm_head:
 * modeling_t5_our.py:39-48,659-671; HF T5Attention / T5DenseReluDense). C[M,N] = epilogue(A[M,K] * B[N,K]^T) on tcgen05;
 * an operand flagged *_mn_major is stored transposed ([K,M] / [K,N]). epi: 0 bf16, 1 relu->bf16, 2 fp32 residual add (R),
 * 3 fp32 atomic accumulate (split-K), 4 relu-backward mask (R = the u32 sign bitmask [M, ceil(N/32)] that epi 1 wrote),  5 fp32,
 * 6 fused row argmax (no C matrix: C = float [M, ldc] per-tile maxima, R = int32 [M, ldr] their columns, slot = 2 * (column / 256)
 * + epilogue-warp group; first maximum = lowest index among equals; 256-wide tiles only).
 * force_bn: 0 = cost model, 64/128/256 = single-CTA tile width, 512 = 256x256 CTA-pair tile (cta_group::2).                 */
/* Several weight gradients in ONE launch (the decoder's six dW = dY^T X per layer, each too small to fill the machine: replaces
 * the autograd-generated per-Linear sgemm calls of T5Attention / T5DenseReluDense backward, hf modeling_t5.py via
 * modeling_t5_our.py:659-671): problem i is C[i][M[i], N[i]] (+)= A[i]^T B[i] with A[i] stored [K, M[i]] and B[i] stored [K, N[i]]
 * (bf16, pitches lda / ldb), C fp32 with pitch ldc[i]; n <= 8; epi 3 = accumulate (red.global.add), 5 = store.                */
int vqacl_gemm_bf16_grouped_mn(int n, const void* const* A, const int* lda, const void* const* B, const int* ldb, void* const* C,
                               const int* ldc, const int* M, const int* N, int K, int epi, float alpha, void* stream);
int vqacl_gemm_bf16(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, void* C, int ldc,
                    const void* R, int ldr, int M, int N, int K, int epi, float alpha, int splits, int force_bn, void* stream);
/* same with the dropout that nn.Dropout applies after the activation / before the residual add (HF T5LayerFF / T5LayerSelfAttention)
 * fused into epilogues 1 and 2: drop_thr16 = round(p * 65536), inv_keep = 1 / (1 - p), drop_key = per-launch 32-bit key.      */
int vqacl_gemm_bf16_ex(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, void* C, int ldc,
                       const void* R, int ldr, int M, int N, int K, int epi, float alpha, int splits, int force_bn,
                       uint32_t drop_thr16, float inv_keep, uint32_t drop_key, void* stream);
/* split-K with one fp32 slab per split (the decoder FFN-out form: a consumer adds the slabs in a fixed order, deterministic
 * unlike the atomic epilogue): slab s = C + s * split_stride ([M, N], pitch ldc, split_stride >= M * ldc) receives
 * alpha * A[:, Ks] B[:, Ks]^T over split s's range Ks of 64-deep k-blocks. The requested split count is clamped to the number
 * of k-blocks and rounded so that no split is empty; *n_slabs receives the count used, and slabs past it are not written.   */
int vqacl_gemm_bf16_slabs(const void* A, int lda, int a_mn_major, const void* B, int ldb, int b_mn_major, float* C, int ldc,
                          long long split_stride, int M, int N, int K, float alpha, int splits, int force_bn, int* n_slabs,
                          void* stream);
/* nn.Linear + residual add + the T5LayerNorm that opens the NEXT sub-layer in one launch (HF T5LayerSelfAttention / T5LayerFF
 * followed by the next layer_norm): C(f32)[M,768] = R + A[M,K] B[768,K]^T; n_out(bf16) = C * rsqrt(mean(C^2) + eps) * norm_w.       */
int vqacl_gemm_resid_rmsnorm(const void* A, int lda, const void* B, int ldb, float* C, const float* R, int M, int K,
                             const float* norm_w, float eps, void* n_out_bf16, void* stream);
/* HF T5LayerNorm forward / backward (hf5.5 modeling_t5.py:46-68; used at modeling_t5_our.py:41,47,160 and in every block)  */
int vqacl_rmsnorm_fwd(const float* x, const float* w, void* y_bf16, float* y_f32, int M, float eps, float scale, void* stream);
int vqacl_rmsnorm_bwd(const void* dn_bf16, const float* x, const float* w, const float* g_in, float* g_out, void* gb_out,
                      float* dw, int M, float eps, float scale, void* stream);
/* HF T5Attention core: softmax(Q K^T + relative bias + masks) V, no 1/sqrt(d) scale (hf5.5 modeling_t5.py:277-338), with the
 * bias / mask construction of JointEncoder.forward (modeling_t5_our.py:225-273) and of the decoder stack folded in.
 * rel_mode 0 none, 1 text x text corner (encoder, Lt = text length), 2 everywhere (decoder self). keymask: additive [B,Sk].   */
int vqacl_attention_fwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, void* o, int ldo, float* lse,
                        int B, int H, int Sq, int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt,
                        const float* keymask, int causal, void* stream);
int vqacl_attention_bwd(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, const void* dO, int ldo,
                        const float* lse, void* dq, void* dk, void* dv, int lddq, int lddk, int lddv, int B, int H, int Sq, int Sk,
                        const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt, const float* keymask, int causal,
                        float* d_rel_table, const void* o_saved /* forward output (pitch ldo) or NULL: enables the key-split
                        backward for Sq <= 16 < Sk */, void* stream);
/* same with the dropout on the probabilities (drop_thr16 = round(p * 65536), inv_keep = 1 / (1 - p), drop_key = per-launch
 * 32-bit key; drop_thr16 = 0 disables it) and, forward only, the KV-cache decode form: element strides between batch entries
 * (0 = densely packed, Sq * ld resp. Sk * ld), and q_off = absolute position of query row 0 (0 <= q_off, q_off + Sq <= 64).
 * lse may be NULL in the forward.                                                                                             */
int vqacl_attention_fwd_ex(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, void* o, int ldo, float* lse,
                           int B, int H, int Sq, int Sk, const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt,
                           const float* keymask, int causal, uint32_t drop_thr16, float inv_keep, uint32_t drop_key,
                           int64_t q_bstride, int64_t k_bstride, int64_t v_bstride, int64_t o_bstride, int q_off, void* stream);
int vqacl_attention_bwd_ex(const void* q, const void* k, const void* v, int ldq, int ldk, int ldv, const void* dO, int ldo,
                           const float* lse, void* dq, void* dk, void* dv, int lddq, int lddk, int lddv, int B, int H, int Sq, int Sk,
                           const float* rel_table, const int32_t* rel_bucket, int rel_mode, int Lt, const float* keymask, int causal,
                           float* d_rel_table, const void* o_saved, uint32_t drop_thr16, float inv_keep, uint32_t drop_key,
                           void* stream);
/* SI prototype path (modeling_t5_our.py:583-615): token means of hidden[:, :split] / hidden[:, split:] (:585-588,601-605) */
int vqacl_proto_means(const float* h, int B, int S, int split, float* meanQ, float* meanV, void* stream);
/* VLT5.calculate_current_prototype (modeling_t5_our.py:500-511)                                                              */
int vqacl_proto_scatter_mean(const float* mean, const float* labels, int B, int C, float* proto, float* cnt, void* stream);
/* VLT5.update_prototype (modeling_t5_our.py:465-498) on explicit state buffers                                               */
int vqacl_proto_update(const float* curQ, const float* curV, const float* cntQ, const float* cntV, float* Qproto, float* Vproto,
                       float* numQ, float* numV, int CQ, int CV, int task_id, int first_step_of_task, int has_mem, float alpha,
                       float beta, void* stream);
/* VLT5.cosine_similarity_multi + the torch.cat of modeling_t5_our.py:434-462,615                                             */
int vqacl_proto_retrieve(const float* P, int C, const float* x, int B, void* out_bf16, int out_pitch_rows, int out_row,
                         int64_t* idx, float* out_f32, float* scratch /* [C,768] fp32 */, void* stream);
/* CrossEntropyLoss(ignore_index=-100, reduction='none') over the tied LM head (modeling_t5_our.py:675-686), fwd and grad     */
int vqacl_ce_fwd(const void* logits_bf16, int ld, int M, int V, const int64_t* labels, float* lse, float* loss, void* stream);
int vqacl_ce_bwd(void* logits_bf16, int ld, int M, int V, const int64_t* labels, const float* lse, const float* w, void* stream);
/* VisualEmbedding.forward after the 2048->768 GEMM (modeling_t5_our.py:93-143)                                               */
int vqacl_visual_embed_fwd(const float* featpre, const float* boxes, const float* bf, const float* wf, const float* Wp,
                           const float* bp, const float* wp, const float* img_emb, const float* shared, int V, int B, int N,
                           int S, int L, float eps, float* x, void* stream);
/* Device-side tail of the reference's __getitem__ + collate_fn (vqa_data_memory.py:179-187, 386-393): boxes (x1,y1,x2,y2) in
 * pixels -> divided by (img_w, img_h, img_w, img_h) and clamped to [0,1]; class ids -> one-hot fp32 rows
 * (torch.zeros(B, C).scatter_(1, ids, 1)). boxes_px [B,N,4], img_wh [B,2], cate_ids / ques_ids int64 [B] (NULL: skipped). */
int vqacl_collate_device(const float* boxes_px, const float* img_wh, int B, int N, float* boxes_out, const int64_t* cate_ids,
                         int n_cate, float* cate_onehot, const int64_t* ques_ids, int n_ques, float* ques_onehot, void* stream);
/* VisualEmbedding.forward in ONE launch (north_star: "the 2048->768 feature projection and the 4-d box projection, fused with
 * LayerNorm in one TMA-staged GEMM epilogue"): tcgen05 GEMM of the bf16 RoI features with the rest of the module as a row tail. */
int vqacl_visual_embed_fused(const void* feats_bf16, const void* Wf_bf16, int F, const float* boxes, const float* bf,
                             const float* wf, const float* Wp, const float* bp, const float* wp, const float* img_emb,
                             const float* shared, int V, int B, int N, int S, int L, float eps, float* featpre, float* x, void* stream);
/* transformers-4.2.1 AdamW.step + torch clip_grad_norm_ (trainer_base.py:130-198, vqacl.py:475-482) over a flat range         */
int vqacl_adamw_hf(float* p, const float* g, float* m, float* v, void* p_bf16, int64_t n, int64_t n_decay, float lr, float beta1,
                   float beta2, float eps, float weight_decay, int step, const float* sumsq, float max_norm, void* stream);
int vqacl_grad_sumsq(const float* g, int64_t n, float* partials, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VQACL_B200_H */
