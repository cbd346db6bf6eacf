/*
 * adaptive_b200.h -- C ABI of libadaptive_b200.so (hand-written sm_100a CUDA).
 *
 * Drop-in boundary for the predict()/add_examples() hot path of codelion/adaptive-classifier.
 * The reference has no FFI of its own: the seams are Python object calls into third-party
 * libraries (SURVEY.md section 8(b)).  Every entry point below names the reference call site it
 * replaces (paths relative to /root/reference/).  The ctypes binding a maintainer would add is in
 * INTEGRATION.md; adaptive_classifier_b200/_cabi.py is that binding.
 *
 * Conventions
 *   - plain C types only; `ac_stream_t` is a cudaStream_t passed as void* (NULL = default stream).
 *   - unless a name ends in `_host`, every data pointer is a DEVICE pointer owned by the caller.
 *   - all matrices are row-major, fp32, ids int64 unless stated; no hidden allocation after
 *     `*_create` / explicit workspaces.
 *   - return value: 0 = ok, negative = error (AC_E_*); text via ac_last_error() (thread-local).
 *   - no CPU fallback exists: with no usable sm_100 device every compute call returns AC_E_CUDA.
 */
#ifndef ADAPTIVE_B200_H
#define ADAPTIVE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *ac_stream_t;

enum {
    AC_OK = 0,
    AC_E_INVALID = -1,   /* bad argument (shape, null pointer, k > limit ...) */
    AC_E_CUDA = -2,      /* CUDA runtime / launch failure, or no sm_100 device */
    AC_E_WORKSPACE = -3, /* workspace too small */
    AC_E_UNSUPPORTED = -4
};

int ac_version(void);                 /* ABI version, currently 1 */
const char *ac_last_error(void);      /* thread-local message of the last failing call */
int ac_device_check(void);            /* 0 when the current device is sm_100 (B200), else AC_E_CUDA */


/* ------------------------------------------------------------------------------------------
 * Stage K -- prototype kNN.  Replaces faiss.IndexFlatL2.search at
 *   src/adaptive_classifier/memory.py:110-114 (call sites :34,106,113,114,158,159,164,172,182,190)
 * ------------------------------------------------------------------------------------------ */

/* algo selector for ac_knn_l2_topk */
enum {
    AC_KNN_AUTO = 0,
    AC_KNN_EXACT = 1,   /* fp32 SIMT exact scan + radix select (any k <= AC_KNN_MAX_K)       */
    AC_KNN_TENSOR = 2   /* tcgen05 coarse pass (kind::f16 over the fp16 shadow, or kind::tf32) + exact fp32 re-rank,
                           k <= AC_KNN_TENSOR_MAX_K.  k <= 16: per-query certification against the rigorous coarse
                           error bound; uncertified queries -- and every query when k > 16 -- take a second,
                           device-conditional tensor pass that collects the provable superset {d~ <= tau + 2 eps},
                           re-ranked exactly (indices identical to AC_KNN_EXACT either way; no host sync) */
};
#define AC_KNN_MAX_K 2048
#define AC_KNN_TENSOR_MAX_K 1024

/* bytes of scratch ac_knn_l2_topk needs for these sizes (device memory, 256-byte aligned) */
int ac_knn_workspace_bytes(int B, int64_t N, int D, int k, int algo, size_t *bytes);

/*
 * out_d[B,k] ascending squared-L2 distances, out_i[B,k] int64 row ids (+row_offset); ties -> lower id;
 * when N < k the tail is (+inf, -1)  [IndexFlatL2.search semantics, memory.py:113-114,121].
 * Distances are the exact fp32 lane-ordered sum restated in oracle/knn_oracle.c (bit-identical).
 * p_sqnorm[N] (nullable) = cached ||p||^2 for the tensor path; computed into the workspace if NULL.
 * p_half (nullable) = fp16 shadow copy of P[N,D] (ac_knn_make_shadow): the tensor path then runs its coarse pass as
 *   tcgen05 kind::f16 over 2.N.D bytes (D %% 64 == 0); candidates are still re-ranked on the fp32 rows, so the
 *   result is the same bits either way.
 * stats (nullable, device int32[4], ACCUMULATED): [0] queries that needed the second tensor pass, [1] queries whose
 *   2-eps band overflowed the candidate buffer (their rows of out_d/out_i are NOT exact: the caller must redo them with
 *   AC_KNN_EXACT), [2] max rows collected for one query, [3] searches.  With stats != NULL the call never synchronises
 *   (graph-capturable); with stats == NULL it synchronises once at the end and recomputes overflowed queries itself.
 */
int ac_knn_l2_topk(const float *Q, const float *P, const float *p_sqnorm, const void *p_half,
                   int B, int64_t N, int D, int k,
                   float *out_d, int64_t *out_i, int64_t row_offset,
                   void *workspace, size_t workspace_bytes, int algo, int32_t *stats, ac_stream_t stream);

/* fp16 (RNE) shadow of the prototype matrix for the tensor path's coarse pass; out_half holds N*D halves */
int ac_knn_make_shadow(const float *P, int64_t N, int D, void *out_half, ac_stream_t stream);

/* ||p||^2 per row (fp32), the cache the tensor path consumes */
int ac_row_sqnorm(const float *P, int64_t N, int D, float *out, ac_stream_t stream);

/* multi-shard merge (new: row-sharded index over G GPUs, SURVEY.md section 8(e)); d[G,B,k], i[G,B,k]
 * -> k smallest by (d, i); entries with i < 0 ignored.  Bit-identical to a single-shard search. */
int ac_topk_merge(const float *d, const int64_t *i, int G, int B, int k,
                  float *out_d, int64_t *out_i, ac_stream_t stream);

/* memory.py:117,128-134: scores[b,:] = softmax_k(exp(-d[b,:])); entries with idx < 0 get 0 */
int ac_proto_scores(const float *d, const int64_t *idx, int B, int k, float *scores, ac_stream_t stream);

/* memory.py:149-150 (prototype = mean of the class's retained examples): rows X[n,D] with class id
 * cls[n] in [0,C) -> mean[C,D], count[C]; classes with no rows keep mean = 0 */
int ac_segment_mean(const float *X, const int32_t *cls, int64_t n, int D, int C,
                    float *mean, int32_t *count, ac_stream_t stream);

/* Device-resident maintenance of the per-class example store for a whole add_examples() call (SURVEY.md 8(f) N2).
 * Replaces the per-example sequence memory.py:60-72 (append, prune when over max_examples_per_class) / :196-217
 * (_prune_examples: keep the `cap` embeddings nearest the mean of the cap + 1, list reordered by that distance) /
 * :138-153 (_update_prototype = mean of the retained embeddings).
 *   rows  [n_slots, cap + 1, D]  class stores;  order [n_slots, cap + 1]: a permutation of the physical slots 0..cap per class,
 *   positions [0, count) = the stored rows in list order, positions [count, cap] = free slots;  count [n_slots].
 *   new_rows [*, D]; new_index [n_new]: row numbers of new_rows grouped by touched class, arrival order inside a class;
 *   cls_start [n_touched + 1]: offsets of the groups in new_index;  touched [n_touched]: class slot of every group.
 * One CTA per touched class processes its new examples sequentially (example j sees the list example j - 1 left).
 * Outputs: src_out [n_touched, cap]: provenance of every retained list position (< old count: that position of the old list,
 * >= old count: old count + index of the new example inside its group, -1: empty); proto_out [n_touched, D].
 * workspace: n_touched * D * 8 bytes. */
int ac_memory_append_prune(float *rows, int32_t *order, int32_t *count, int cap, int D, const float *new_rows,
                           const int32_t *new_index, const int32_t *cls_start, const int32_t *touched, int n_touched,
                           int32_t *src_out, float *proto_out, void *workspace, size_t workspace_bytes, ac_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Stage H -- adaptive head.  Replaces nn.Module.__call__ / autograd / AdamW on AdaptiveHead:
 *   forward  src/adaptive_classifier/models.py:71-80, classifier.py:428-442, :1341-1354
 *   training classifier.py:333-351, :1489-1505, multilabel.py:387-397
 * Weights in nn.Linear layout: W0[H0,D], W1[H1,H0], W2[C,H1]  (H0 = D, H1 = D/2 in the reference).
 * ------------------------------------------------------------------------------------------ */
enum { AC_ACT_LOGITS = 0, AC_ACT_SOFTMAX = 1, AC_ACT_SIGMOID = 2 };
enum { AC_LOSS_CE = 0, AC_LOSS_BCE = 1 };

typedef struct {
    int D, H0, H1, C;
    float *W0, *b0, *W1, *b1, *W2, *b2;
} ac_head_params;

/* eval-mode forward (dropout inactive).  out[B,C]; scratch >= B*(H0+H1) floats */
int ac_head_forward(const float *X, int B, const ac_head_params *p, int act,
                    float *out, float *scratch, size_t scratch_floats, ac_stream_t stream);

typedef struct {
    float lr, beta1, beta2, eps, weight_decay, max_norm; /* AdamW + clip_grad_norm_ */
    int step;                /* 1-based count of this update (bias correction) */
    int loss_kind;           /* AC_LOSS_CE: targets int64[B]; AC_LOSS_BCE: targets float[B,C] */
    float dropout_p;         /* 0.1 in the reference; 0 disables */
    const float *mask0;      /* optional injected dropout masks [B,H0], [B,H1] holding 0 or 1/(1-p);   */
    const float *mask1;      /*   NULL -> Philox masks from (seed, step)                                */
    uint64_t seed;
    /* optional EWC term (ewc.py:96-115): grad += 2*lambda/B * F*(theta-theta*) over the first
       ewc_rows_out rows of the output layer (the head may have grown), NULL = off */
    const ac_head_params *ewc_fisher;
    const ac_head_params *ewc_star;
    float ewc_lambda;
    int ewc_C_old;
} ac_train_cfg;

/* bytes of workspace for a training / gradient call with `batch` rows per step and n_steps steps (1 for a single step) */
int ac_head_train_workspace_bytes(int batch, int n_steps, const ac_head_params *p, size_t *bytes);

/* one optimizer step: fwd(train) + loss + bwd + [EWC grad] + global-norm clip + AdamW, as one launch of the persistent
 * cooperative kernel of csrc/head_train.cuh (B <= 64; D, H0, H1 multiples of 4).
 * m, v: AdamW moments (same shapes as p).  out_stats[0] = task loss, [1] = ewc penalty,
 * [2] = grad norm before clipping (device floats). */
int ac_head_train_step(const float *X, const void *targets, int B,
                       ac_head_params *p, ac_head_params *m, ac_head_params *v,
                       const ac_train_cfg *cfg, float *out_stats,
                       void *workspace, size_t workspace_bytes, ac_stream_t stream);

/* one EPOCH of the reference's training loops (classifier.py:329-353, :1485-1507; multilabel.py:381-399) in one call:
 * X[n,D], targets (int64[n] or float[n,C]) and the shuffled index list perm[n] (what the reference's DataLoader with
 * torch.Generator().manual_seed(42) yields) live on the device; batches of `batch` rows (last one partial) are gathered
 * and stepped inside ONE kernel launch (the grid stays resident for the whole epoch: parameters live in shared memory, six
 * grid barriers per step).  cfg->step = 1-based number of the first update.  loss_accum (nullable): [0] += task loss + EWC
 * penalty per step.  step_stats (nullable): [ceil(n / batch), 3] = (task loss, EWC penalty, grad norm before clipping) of
 * every step -- what the reference's loop reads back with loss.item() (classifier.py:353, :1507).
 * workspace: ac_head_train_workspace_bytes(batch, ceil(n / batch), ...). */
int ac_head_train_epoch(const float *X, const void *targets, const int64_t *perm, int n, int batch,
                        ac_head_params *p, ac_head_params *m, ac_head_params *v, const ac_train_cfg *cfg,
                        float *loss_accum, float *step_stats, void *workspace, size_t workspace_bytes, ac_stream_t stream);

/* diagnostic: per-phase time of the training kernel: nanoseconds three observed CTAs (one per layer of the head) spent in each
 * of the 7 phases and 6 grid barriers of a step (13 counters) and inside the product routines (7 counters from index 14), summed
 * over all steps since enabled.  enable != 0 starts accumulating; out72_host (nullable) receives 3 x 24 counters. */
int ac_head_phase_timing(int enable, unsigned long long *out72_host);
/* diagnostic: launch plan of the training kernel: out5 = {CTAs, operand-ring stages, AdamW moments resident in shared memory (0/1),
 * dynamic shared-memory bytes, reserved} */
int ac_head_train_plan(int batch, const ac_head_params *p, int *out5);

/* gradient only (no update) of mean CE/BCE wrt all parameters, eval mode: the building block of
 * EWC._compute_fisher (ewc.py:67-92).  fisher += grad^2 * inv_n_batches when fisher != NULL */
int ac_head_grad(const float *X, const void *targets, int B, const ac_head_params *p, int loss_kind,
                 ac_head_params *grad_out, ac_head_params *fisher_accum, float inv_n_batches,
                 float *out_loss, void *workspace, size_t workspace_bytes, ac_stream_t stream);

/* ewc.py:105-115: out[0] = lambda/bs * sum F*(theta-theta*)^2 over the parameters (C_old rows of the
 * output layer) */
int ac_ewc_penalty(const ac_head_params *p, const ac_head_params *fisher, const ac_head_params *star,
                   float lambda, float inv_batch, int C_old, float *out, ac_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Stage E -- encoder.  Replaces `self.model(**inputs).last_hidden_state[:,0,:]` + F.normalize at
 *   src/adaptive_classifier/classifier.py:1271-1275 (HF BertModel / RobertaModel forward).
 * ------------------------------------------------------------------------------------------ */
enum { AC_ARCH_BERT = 0, AC_ARCH_ROBERTA = 1, AC_ARCH_MODERNBERT = 2 };
enum {
    AC_PREC_TF32 = 0,   /* tcgen05 kind::tf32 on fp32 storage (kNN coarse pass, ac_linear_tc tests) */
    AC_PREC_F16 = 1     /* tcgen05 kind::f16 with fp16 operands (RNE from fp32; same 10-bit mantissa as tf32),
                           fp32 accumulation; the encoder's precision: 1.7e-4 on distances, bf16 would be 1.4e-3 */
};

typedef struct {
    int arch;            /* AC_ARCH_* */
    int layers, hidden, heads, intermediate;
    int vocab, max_pos, type_vocab;
    int pad_idx;         /* roberta: position ids start at pad_idx+1 */
    float ln_eps;
    int precision;       /* AC_PREC_* */
    int max_tokens;      /* workspace is sized for B*S <= max_tokens */
    int cls_only;        /* != 0: the last layer's output projection / FFN / LayerNorms run on the CLS rows only
                            (classifier.py:1272 uses nothing else); 0 keeps the full last hidden state */
} ac_encoder_config;

/* device pointers to the HF state_dict tensors (fp32, HF layout [out,in]) */
typedef struct {
    const float *word_emb, *pos_emb, *type_emb, *emb_ln_w, *emb_ln_b;
    /* arrays of `layers` device pointers each (host arrays of device pointers) */
    const float *const *q_w, *const *q_b, *const *k_w, *const *k_b, *const *v_w, *const *v_b;
    const float *const *ao_w, *const *ao_b, *const *ao_ln_w, *const *ao_ln_b;
    const float *const *ff1_w, *const *ff1_b, *const *ff2_w, *const *ff2_b;
    const float *const *out_ln_w, *const *out_ln_b;
} ac_encoder_weights;

typedef struct ac_encoder ac_encoder;

/* copies + repacks the weights (fused QKV, operand rounding) and allocates the activation workspace */
int ac_encoder_create(const ac_encoder_config *cfg, const ac_encoder_weights *w, ac_encoder **out);
int ac_encoder_destroy(ac_encoder *enc);

/* ModernBERT (the reference's tests use answerdotai/ModernBERT-base: tests/test_order_independence.py:10,
 * tests/test_confidence_consistency.py:14), HF transformers models/modernbert/modeling_modernbert.py:
 *   embeddings LayerNorm(tok_embeddings[ids]) :52-71; pre-LN block x += Wo(attn(attn_norm(x))), x += mlp(mlp_norm(x))
 *   :313-343 (attn_norm = identity in layer 0); fused Wqkv [3H, H] with RoPE (rotate_half, pairs d and d + 32 of each
 *   64-wide head) :204-310; GeGLU mlp Wo(gelu_erf(input) * gate) with input, gate = Wi(x).chunk(2) :74-91; final_norm.
 * Sliding layers see key k from query q iff |q - k| <= window (inclusive, masking_utils.py:121-131).  Creates the same
 * ac_encoder handle as ac_encoder_create: forward_cls, last_hidden, destroy and the pipeline take it unchanged, and
 * forward_cls ignores type_ids for it (ModernBERT has no token types).  S <= 512, head_dim 64. */
typedef struct {
    int layers, hidden, heads;
    int intermediate;        /* I: Wi has 2I rows, mlp.Wo has I columns; multiple of 64 */
    int vocab;
    float norm_eps;
    int precision;           /* AC_PREC_F16 */
    int max_tokens;
    int cls_only;            /* as in ac_encoder_config */
    const int *window;       /* host array [layers]: key window of each layer (config.sliding_window), 0 = global */
    const float *rope_theta; /* host array [layers]: rope_theta of each layer's type */
} ac_modernbert_config;

/* device pointers to the HF state_dict tensors (fp32, [out, in]); a NULL bias (or NULL bias array) means zero */
typedef struct {
    const float *tok_emb, *emb_norm_w, *emb_norm_b;
    /* arrays of `layers` device pointers each (host arrays); attn_norm_w[0] / attn_norm_b[0] are ignored (NULL) */
    const float *const *attn_norm_w, *const *attn_norm_b;
    const float *const *Wqkv, *const *Wqkv_b, *const *Wo, *const *Wo_b;
    const float *const *mlp_norm_w, *const *mlp_norm_b;
    const float *const *Wi, *const *Wi_b, *const *mlp_Wo, *const *mlp_Wo_b;
    const float *final_norm_w, *final_norm_b;
} ac_modernbert_weights;

int ac_encoder_create_modernbert(const ac_modernbert_config *cfg, const ac_modernbert_weights *w, ac_encoder **out);

/* ids[B,S] int32 token ids, mask[B,S] int32 (1 keep / 0 pad; NULL = all ones), type_ids nullable.
 * out_unit_cls[B,H] = L2-normalised (eps 1e-12) CLS row of the last hidden state. */
int ac_encoder_forward_cls(ac_encoder *enc, const int32_t *ids, const int32_t *mask,
                           const int32_t *type_ids, int B, int S, float *out_unit_cls,
                           ac_stream_t stream);


/* debugging / parity: copy the full last hidden state [B*S,H] of the previous forward */
int ac_encoder_last_hidden(ac_encoder *enc, float *out, int64_t n_floats, ac_stream_t stream);

/* generic tensor-core linear (the encoder's GEMM with its fused epilogues), exposed for parity tests and roofline
 * measurement: Y[M,N] = epi(X[M,K] W[N,K]^T + bias) (+ residual).  epi: 0 bias, 1 bias+GELU(erf), 2 bias+fp32 residual.
 * precision AC_PREC_TF32: X, W, Y fp32 (operands used as stored; round_out != 0 rounds Y to tf32);
 * precision AC_PREC_F16 : X, W fp16, Y fp32 or (out_half != 0, epi != 2) fp16. */
int ac_linear_tc(const void *X, const void *W, const float *bias, const float *residual, void *Y,
                 int M, int N, int K, int epi, int round_out, int precision, int out_half, ac_stream_t stream);

/* the encoder's attention, exposed for parity tests; it runs the same dispatch ac_encoder_forward_cls uses (S <= 128 kernel or
 * the 128-query-block kernel, windowed when 0 < window < S - 1).  Per (sequence b, head h), H = 64 * heads:
 *   ctx[b*S + q, 64h + :] = sum_k P[q,k] V[k] / sum_k P[q,k],  P[q,k] = exp((Q[q].K[k] - max) / 8) over the keys k < S with
 *   mask[b,k] != 0 and, when windowed, |q - k| <= window; a query row with no such key gets zeros.
 * qk  fp16 [qk_rows, 2H]: Q in columns [0, H), K in [H, 2H) (the encoder's layout); qk_rows >= B*S.  The kernels read whole
 *     128-row tiles, so rows of neighbouring sequences and rows past B*S are loaded and must be ignored.
 * vT  fp16 [(b, h, d), S_pad]: V transposed per (sequence, head), S_pad = roundup(S, 8); keys S .. S_pad-1 are ignored.
 * mask int32 [B, S] nullable (1 keep / 0 pad), window 0 = global, ctx fp16 [B*S, H], S <= 512. */
int ac_attention(const void *qk, int64_t qk_rows, const void *vT, const int32_t *mask, int B, int S, int heads, int window,
                 void *ctx, ac_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * predict_batch() glue on the device (classifier.py:1329-1384) and the end-to-end pipeline.
 * ------------------------------------------------------------------------------------------ */

/* memory.py:117-134 generalised to many rows per class (SURVEY.md section 8(d)): the k nearest rows (d asc, idx)
 * are mapped through row_class[global row id] (NULL: class = row id), a class keeps its nearest row,
 * out_score = softmax(exp(-d)) over the distinct classes; tails padded with (-1, 0).  k <= 32. */
int ac_proto_class_scores(const float *d, const int64_t *idx, const int32_t *row_class, int B, int k,
                          int32_t *out_cls, float *out_score, ac_stream_t stream);

/* the same for k up to 1024 (predict(): k = num_classes, classifier.py:424-425); class ids < n_classes <= 4096 */
int ac_proto_class_scores_n(const float *d, const int64_t *idx, const int32_t *row_class, int B, int k, int n_classes,
                            int32_t *out_cls, float *out_score, ac_stream_t stream);

/* predict() blend over ALL classes (classifier.py:446-480): combined[c] = proto_score[c] * w_proto[c] + head_probs[b,c] *
 * w_head[c] (per-class weights from training_history: < 10 examples -> 0.3 / 0.7, else 0.7 / 0.3), normalised by the sum,
 * top kout.  proto_cls / proto_score [B, kp] as written by ac_proto_class_scores(_n); head_probs [B, C] nullable. */
int ac_blend_dense(const int32_t *proto_cls, const float *proto_score, int kp, const float *head_probs, int B, int C,
                   const float *w_proto, const float *w_head, int kout, int32_t *out_cls, float *out_score, ac_stream_t stream);

/* classifier.py:1347-1350 (torch.topk of the head probabilities): out_neg_vals[B,k] holds the k largest values
 * NEGATED (ascending), out_idx[B,k] their column ids; ties -> lower id. */
int ac_topk_desc_workspace_bytes(int B, int C, int k, size_t *bytes);
int ac_topk_desc(const float *values, int B, int C, int k, float *out_neg_vals, int64_t *out_idx,
                 void *workspace, size_t workspace_bytes, ac_stream_t stream);

/* classifier.py:1358-1384: combined[label] = w_proto*proto + w_head*head, stable descending sort,
 * normalised by the sum, top k.  head_neg_val as produced by ac_topk_desc.  k, kh <= 32. */
int ac_blend_topk(const int32_t *proto_cls, const float *proto_score, const int64_t *head_idx,
                  const float *head_neg_val, int B, int k, int kh, float w_proto, float w_head,
                  int32_t *out_cls, float *out_score, ac_stream_t stream);

/* E -> K -> class scores -> H -> top-k -> blend with all intermediate buffers owned by the handle.
 * head may be NULL (prototype-only prediction).  row_class nullable. */
typedef struct ac_pipeline ac_pipeline;
int ac_pipeline_create(ac_encoder *enc, const float *P, const float *p_sqnorm, const void *p_half,
                       const int32_t *row_class, int64_t N, int D, const ac_head_params *head, int max_B, int S, int k,
                       int64_t row_offset, int shards /* 1, or the number of GPUs the rows are sharded over */, ac_pipeline **out);
int ac_pipeline_destroy(ac_pipeline *pl);
/* device buffers at the boundary (bench.py `value`) */
int ac_pipeline_predict_device(ac_pipeline *pl, const int32_t *ids_dev, const int32_t *mask_dev, int B,
                               int32_t *out_cls_dev, float *out_score_dev, ac_stream_t stream);
/* HOST buffers at the boundary (bench.py `e2e`): H2D of ids and D2H of the [B,k] result inside the call.  The device part of the
 * step is replayed as a CUDA graph from the third call with a batch size on (first: ordinary launches, second: capture) -- at B = 1
 * the ~110 launches of a step cost more host time than GPU time (0.92 instead of 1.15 ms per query).  Results are identical to the
 * eager step; AC_PIPELINE_GRAPH=0 in the environment, or enabled per-kernel profiling (ac_profile_enable), keeps the step eager. */
int ac_pipeline_predict_host(ac_pipeline *pl, const int32_t *ids_host, int B, int32_t *out_cls_host,
                             float *out_score_host, ac_stream_t stream);
/* The phases of one step, for the row-sharded multi-GPU search (SURVEY.md section 8(e)): the caller (parallel.py) runs the
 * two collectives between them on the same stream -- all-gather of the unit embeddings, ONE all-to-all of the packed
 * (distance, id) candidates -- so that N > 1 executes the same kernels, with the same side-stream overlap of the head, as N = 1.
 *   ac_pipeline_encode         ids -> unit CLS rows (ac_pipeline_embeddings returns the device pointer, [B, D])
 *   ac_pipeline_search_shard   q_all[G*B, D] (rank-major) over THIS shard -> packed: G chunks of (d[B,k] fp32 | id[B,k] int64)
 *   ac_pipeline_finish_sharded received chunks (chunk g = shard g's candidates of MY queries) -> merge by (d, global id)
 *                              [bit-identical to the unsharded search] -> class scores -> head -> blend */
int ac_pipeline_encode(ac_pipeline *pl, const int32_t *ids_dev, const int32_t *mask_dev, int B, ac_stream_t stream);
int ac_pipeline_embeddings(ac_pipeline *pl, const float **emb_dev);
int ac_pipeline_search_shard(ac_pipeline *pl, const float *q_all, int G, int B, void *packed, ac_stream_t stream);
int ac_pipeline_finish_sharded(ac_pipeline *pl, const void *received, int G, int B, int32_t *out_cls_dev, float *out_score_dev,
                               ac_stream_t stream);
/* search statistics accumulated since the last reset (synchronises): see ac_knn_l2_topk `stats` */
int ac_pipeline_knn_stats(ac_pipeline *pl, int32_t *out4_host, int reset, ac_stream_t stream);
/* parity tests: copy the last call's unit CLS rows [B,D] and kNN result [B,k] into caller device buffers */
int ac_pipeline_debug_copy(ac_pipeline *pl, int B, float *emb_out, float *knn_d_out, int64_t *knn_i_out,
                           ac_stream_t stream);

/* ------------------------------------------------------------------------------------------
 * Measurement hooks (bench.py): number of kernels launched by this library so far, and optional
 * CUDA-event timing of the dominant kernels on their launching stream.
 * classes: 0 encoder tcgen05 GEMM, 1 attention, 2 kNN tensor pass 1, 3 kNN exact scan, 4 kNN tensor pass 2 (device-conditional)
 * ------------------------------------------------------------------------------------------ */
long long ac_launch_count(void);
int ac_profile_enable(int on);
int ac_profile_read(int cls, double *ms, double *flops, double *bytes, long long *launches);

#ifdef __cplusplus
}
#endif
#endif /* ADAPTIVE_B200_H */
