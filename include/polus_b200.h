/*
 * libpolus_b200.so -- C ABI of the B200-native polus training step.
 *
 * The reference (bioinformatics-ua/polus) has no FFI: its device work is TensorFlow / HuggingFace /
 * tensorflow_addons / Horovod library calls made from Python (SURVEY.md section 8b).  Each entry point
 * below therefore cites the *reference call site* whose device work it replaces.  The Python host
 * (the polus_b200 package) binds these with ctypes; nothing here takes or returns a torch / numpy type.
 *
 * Conventions
 *   - every function returns 0 on success or a negative polus_status_t; polus_last_error() gives
 *     the thread-local message (reference raises Python exceptions: polus/training.py:59-60,251,257).
 *   - pointers named d_* are device pointers, h_* host pointers; `stream` is a cudaStream_t (or NULL).
 *   - activations are row-major; "bf16" is __nv_bfloat16 storage; all reductions are fp32.
 *   - one process per GPU, calls made from one host thread (polus/__init__.py:122).
 */
#ifndef POLUS_B200_H
#define POLUS_B200_H
#include <stdint.h>
#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    POLUS_OK = 0,
    POLUS_ERR_INVALID = -1,
    POLUS_ERR_CUDA = -2,
    POLUS_ERR_NCCL = -3,
    POLUS_ERR_OOM = -4,
    POLUS_ERR_SHAPE = -5
} polus_status_t;

typedef enum { POLUS_F32 = 0, POLUS_BF16 = 1, POLUS_I32 = 2, POLUS_U8 = 3 } polus_dtype_t;
typedef uint16_t polus_bf16_t; /* __nv_bfloat16 storage */

typedef enum {
    POLUS_ACT_NONE = 0,
    POLUS_ACT_GELU = 1, /* exact erf GELU: HF BertIntermediate, hidden_act="gelu" */
    POLUS_ACT_RELU = 2, /* tutorials/classifier_example.py:46 */
    POLUS_ACT_SWISH = 3, /* polus/ner/models.py:30 */
    POLUS_ACT_TANH = 4, /* HF BertPooler */
    POLUS_ACT_MISH = 5, /* polus/models.py:53-57 */
    POLUS_ACT_DERIV = 100, /* polus_act_bwd_colsum only: `z` already holds act'(pre-activation) (polus_gemm_t.c2_kind = 1) */
    POLUS_ACT_DERIV_U8 = 101 /* ... as 8-bit fixed point, one byte per element: gelu' = (q - 28) * 0.005 (c2_kind = 2) */
} polus_act_t;

/* ---------------------------------------------------------------- runtime / memory ---------- */
/* replaces: TF device placement + allocator (polus/__init__.py:107-122) */
const char* polus_last_error(void);
int polus_version(void);
int polus_init(int device);                 /* cudaSetDevice + capability check (sm_100) */
int polus_device_count(int* n);
int polus_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* total_mem);
int polus_malloc(void** d_ptr, size_t bytes);
int polus_free(void* d_ptr);
int polus_host_alloc(void** h_ptr, size_t bytes);   /* pinned */
int polus_host_free(void* h_ptr);
int polus_memcpy_h2d(void* d_dst, const void* h_src, size_t bytes, void* stream);
int polus_memcpy_d2h(void* h_dst, const void* d_src, size_t bytes, void* stream);
int polus_memcpy_d2d(void* d_dst, const void* d_src, size_t bytes, void* stream);
int polus_memset(void* d_ptr, int value, size_t bytes, void* stream);
int polus_stream_create(void** stream, int high_priority);  /* 0 normal, 1 highest (collectives), 2 background */
int polus_stream_destroy(void* stream);
int polus_stream_sync(void* stream);
int polus_device_sync(void);
int polus_event_create(void** event);
int polus_event_destroy(void* event);
int polus_event_record(void* event, void* stream);
int polus_event_sync(void* event);
int polus_event_elapsed_ms(void* start, void* stop, float* ms);
int polus_stream_wait_event(void* stream, void* event);
/* CUDA-graph capture of one train_step: replaces the tf.function graph of
 * polus/training.py:150-151 (trace once per input signature, replay afterwards). */
int polus_graph_begin(void* stream);
int polus_graph_end(void* stream, void** graph_exec);
int polus_graph_launch(void* graph_exec, void* stream);
int polus_graph_destroy(void* graph_exec);
/* number of kernels launched by this library since process start (bench.py "gpu_launches") */
int64_t polus_launch_count(void);
/* NVTX-free profiler window: cudaProfilerStart/Stop (polus/callbacks.py:408-470 Profiler) */
int polus_profiler_start(void);
int polus_profiler_stop(void);
/* per-step profiler ranges: tf.profiler.experimental.Trace('step', step_num=n) of polus/callbacks.py:442-470 (NVTX
 * push / pop on the calling thread; visible to nsys / ncu --nvtx, free when no profiler is attached) */
int polus_profiler_range_push(const char* name);
int polus_profiler_range_pop(void);

/* ---------------------------------------------------------------- dense contractions -------- */
/* One operand of a (batched) GEMM.  `mn_major` = 0: the reduction dim K is contiguous
 * (row r of length K at ptr + r*ld); 1: the M (or N) dim is contiguous (row k of length MN at
 * ptr + k*ld).  Batch index = b1 * batch0 + b0, element offset b0*bs0 + b1*bs1. */
typedef struct {
    const void* ptr;
    int64_t ld;       /* elements */
    int64_t bs0, bs1; /* elements */
    int32_t mn_major;
    int32_t dtype; /* polus_dtype_t; the tcgen05 path needs POLUS_BF16 */
} polus_operand_t;

typedef struct {
    int32_t M, N, K;
    int32_t batch0, batch1; /* >= 1 */
    polus_operand_t A;      /* [M,K] */
    polus_operand_t B;      /* [N,K] */
    void* C;                /* [M,N] row-major */
    int64_t ldc, cbs0, cbs1;
    int32_t c_dtype;   /* POLUS_BF16 or POLUS_F32 */
    void* C2;          /* optional: pre-activation copy (same layout/dtype as C), may be NULL */
    const float* bias; /* optional [N] fp32 */
    float alpha;       /* C = act(alpha * A.B^T + bias) */
    int32_t act;       /* polus_act_t */
    int32_t accumulate; /* 1: C += result (fp32 C only; required when split_k > 1) */
    int32_t split_k;    /* >= 1 */
    /* Fused backward of an activation layer (tcgen05 path, bf16 C).  Forward: c2_kind = 1 stores act'(pre-activation)
     * in C2 instead of the pre-activation itself.  Backward (dgrad of the NEXT layer): Emul = that tensor, same
     * layout as C, multiplies the result element-wise, C = (alpha A.B^T + bias) * Emul, and colsum[n] += sum_m C[m,n]
     * accumulates the bias gradient (fp32 atomics) -- the tf.GradientTape ops GeluGrad + BiasAddGrad of
     * polus/training.py:185 without a pass over the [M,N] tensor. */
    int32_t c2_kind;    /* 0: C2 = pre-activation, 1: C2 = activation derivative (bf16), 2: C2 (GELU forward) / Emul (the
                         * dgrad that consumes it) = gelu' as 8-bit fixed point, one byte per element, row pitch ldc BYTES,
                         * q = 28 + round(200 gelu'): half the bytes of these two store-bandwidth-bound GEMMs; supported
                         * where polus_gemm_tc_supported says so (256-wide pair tiles, N % 32 == 0, ldc % 16 == 0) */
    const void* Emul;   /* optional [M,N] multiplier, bf16 (or 8-bit, c2_kind = 2), ldc/cbs0/cbs1 as C; requires act == NONE, no C2 */
    float* colsum;      /* optional fp32 [N] */
} polus_gemm_t;

/* tcgen05 / TMEM / TMA GEMM.  Replaces the cuBLAS calls TF makes for HF TFBertLayer's Dense
 * layers and batched attention matmuls (polus/models.py:205-213), the NER head Dense
 * (polus/ner/models.py:36) and all their gradients (polus/training.py:185). */
int polus_gemm_tc(const polus_gemm_t* g, void* stream);
/* CUDA-core GEMM for shapes a tcgen05 tile cannot take (N=4 tag projection, N=10 tutorial head)
 * and the on-device checker for polus_gemm_tc in tests.  Accepts F32 or BF16 operands. */
int polus_gemm_small(const polus_gemm_t* g, void* stream);
/* Narrow dense layer, N <= 32 (polus/ner/models.py:37 tag projection; tutorials/classifier_example.py:47):
 * y = act(x.W + b) with W [K,N] fp32; x f32 or bf16; optional z = pre-activation.  One pass over x. */
int polus_skinny_supported(int K, int N);
int polus_skinny_fwd(const void* d_x, int x_dtype, const float* d_W, const float* d_b, int M, int K, int N,
                     int act, float* d_y, float* d_z, void* stream);
/* dx = dz.W^T (may be NULL), gW += x^T.dz, gb += colsum(dz) (may be NULL) */
int polus_skinny_bwd(const void* d_x, int x_dtype, const float* d_W, const float* d_dz, int M, int K, int N,
                     void* d_dx, int dx_dtype, float* d_gW, float* d_gb, void* stream);
/* 1 if polus_gemm_tc accepts this problem (alignment / dtype rules), else 0.  N % 8 != 0 (vocabulary projections) is
 * accepted for plain and bias-only problems with a K-major B (from polus_version() 103).  The contents of C's columns
 * N .. ldc are unspecified: readers must not use them. */
int polus_gemm_tc_supported(const polus_gemm_t* g);

/* ---------------------------------------------------------------- memory-bound encoder ops -- */
/* Dropout sites are addressed by (seed, site, *d_step): Philox4x32-10 counters, no stored masks. */

/* HF TFBertEmbeddings (polus/data.py:526-545, models.py:225): y = LN(word[ids]+pos[s]+type[tt]),
 * then dropout.  Saves xhat-free stats (mean, rstd) and the pre-LN sum z for backward. */
int polus_embed_ln_fwd(const int32_t* d_ids, const int32_t* d_tt, const float* d_word,
                       const float* d_pos, const float* d_type, const float* d_gamma,
                       const float* d_beta, int B, int S, int H, int vocab, int n_types, float eps,
                       float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                       polus_bf16_t* d_y, float* d_z, float* d_mean, float* d_rstd, void* stream);
int polus_embed_ln_bwd(const polus_bf16_t* d_dy, const float* d_z, const float* d_mean,
                       const float* d_rstd, const float* d_gamma, const int32_t* d_ids,
                       const int32_t* d_tt, int B, int S, int H, int vocab, int n_types, float p_drop,
                       uint64_t seed, uint32_t site, const uint32_t* d_step, float* d_gword,
                       float* d_gpos, float* d_gtype, float* d_ggamma, float* d_gbeta, float* d_ws,
                       void* stream);
size_t polus_embed_ws_floats(int B, int S, int H); /* size of d_ws above */
/* The same with per-token position ids (RoBERTa family, or explicit ids): the position row of token (b, s) is
 * d_pos_ids[b*S + s], clamped to the n_pos rows of d_pos.  Backward adds position gradients keyed by that id; the
 * padding_idx row receives the gradients of pad tokens (TF semantics).  Available from polus_version() 102. */
int polus_embed_ln_fwd_pos(const int32_t* d_ids, const int32_t* d_tt, const float* d_word,
                           const float* d_pos, const float* d_type, const float* d_gamma,
                           const float* d_beta, int B, int S, int H, int vocab, int n_types, float eps,
                           float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                           polus_bf16_t* d_y, float* d_z, float* d_mean, float* d_rstd,
                           const int32_t* d_pos_ids, int n_pos, void* stream);
int polus_embed_ln_bwd_pos(const polus_bf16_t* d_dy, const float* d_z, const float* d_mean,
                           const float* d_rstd, const float* d_gamma, const int32_t* d_ids,
                           const int32_t* d_tt, int B, int S, int H, int vocab, int n_types, float p_drop,
                           uint64_t seed, uint32_t site, const uint32_t* d_step, float* d_gword,
                           float* d_gpos, float* d_gtype, float* d_ggamma, float* d_gbeta, float* d_ws,
                           const int32_t* d_pos_ids, int n_pos, void* stream);
/* HF create_position_ids_from_input_ids on the device: d_pos[b,s] = padding_idx + #(d_ids[b,0..s] != padding_idx)
 * where d_ids[b,s] != padding_idx, else padding_idx.  [B,S] int32 in and out; no host round trip. */
int polus_position_ids(const int32_t* d_ids, int B, int S, int padding_idx, int32_t* d_pos, void* stream);

/* HF TFBertSelfOutput / TFBertOutput: y = LN(dropout(x) + res), eps 1e-12.  x is overwritten with
 * z = dropout(x)+res (kept for backward).  res may be NULL. */
int polus_ln_res_fwd(polus_bf16_t* d_x_inout, const polus_bf16_t* d_res, const float* d_gamma,
                     const float* d_beta, int M, int H, float eps, float p_drop, uint64_t seed,
                     uint32_t site, const uint32_t* d_step, polus_bf16_t* d_y, float* d_mean,
                     float* d_rstd, uint8_t* d_keepbits, void* stream);
/* d_keepbits (may be NULL): [M * H/8] bytes, the dropout decisions of this call (bit j of byte c = element 8c+j kept);
 * handing them to polus_ln_res_bwd saves it the Philox regeneration. */
/* d(y) = d_dy (+ d_dy2 when not NULL: a second contribution from the residual stream, summed in-kernel).
 * Writes d_dx (through dropout) and d_dres (may be NULL; may alias d_dx when p_drop == 0); dgamma/dbeta are
 * accumulated; d_gbias_x (may be NULL) also receives the column sums of d_dx, i.e. the bias gradient of the Dense
 * layer that produced x, saving that layer a separate reduction pass.  d_keepbits: the forward call's dropout
 * decisions, or NULL to regenerate them from (seed, site, *d_step). */
int polus_ln_res_bwd(const polus_bf16_t* d_dy, const polus_bf16_t* d_dy2, const polus_bf16_t* d_z,
                     const float* d_mean, const float* d_rstd, const float* d_gamma, int M, int H, float p_drop,
                     uint64_t seed, uint32_t site, const uint32_t* d_step, polus_bf16_t* d_dx,
                     polus_bf16_t* d_dres, float* d_ggamma, float* d_gbeta, float* d_gbias_x,
                     const uint8_t* d_keepbits, void* stream);
size_t polus_ln_ws_floats(int H);

/* HF TFBertSelfAttention softmax: P = softmax(scores*scale + (1-mask)*-10000) (polus/models.py:
 * 175-195), Pd = dropout(P).  scores bf16 [rows = B*nh*S, S]; mask int32 [B,S] or NULL.
 * d_p receives P; d_pd receives Pd (may alias d_p when p_drop == 0). */
int polus_softmax_fwd(const polus_bf16_t* d_scores, const int32_t* d_mask, int B, int nh, int Sq,
                      int Sk, float scale, float p_drop, uint64_t seed, uint32_t site,
                      const uint32_t* d_step, polus_bf16_t* d_p, polus_bf16_t* d_pd, void* stream);
/* dS = scale * P o (dP - sum_j P dP) with dP = dropout-bwd(dPd); writes dS over d_dpd_inout and,
 * when p_drop > 0, Pd over d_p_inout (needed by the dV GEMM). */
int polus_softmax_bwd(polus_bf16_t* d_p_inout, polus_bf16_t* d_dpd_inout, int B, int nh, int Sq, int Sk,
                      float scale, float p_drop, uint64_t seed, uint32_t site,
                      const uint32_t* d_step, void* stream);

/* Fused self-attention core for head_dim 64, S <= 512 (S % 32 == 0) on the packed projection qkv [B,S,3*nh*64]
 * (q|k|v column blocks): ctx = dropout(softmax(QK^T/8 + (1-mask)*-10000)) V, scores/probabilities kept in
 * TMEM/shared memory.  Saves lse [B,nh,S] (row log-sum-exp) for the backward, which recomputes P.
 * Replaces HF TFBertSelfAttention's matmul/softmax/dropout/matmul and their gradients (polus/models.py:175-213). */
int polus_attention_supported(int S, int head_dim);           /* head_dim 64, 32 <= S <= 512, S % 32 == 0 */
size_t polus_attention_keepbits_words(int B, int S, int nh);   /* uint32 words of the dropout keep-bit buffer */
int polus_attention_fwd(const polus_bf16_t* d_qkv, const int32_t* d_mask, int B, int S, int nh, int head_dim,
                        float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step, polus_bf16_t* d_ctx,
                        float* d_lse, uint32_t* d_keepbits, void* stream);
int polus_attention_bwd(const polus_bf16_t* d_qkv, const int32_t* d_mask, const polus_bf16_t* d_ctx,
                        const polus_bf16_t* d_dctx, const float* d_lse, int B, int S, int nh, int head_dim,
                        float p_drop, uint64_t seed, uint32_t site, const uint32_t* d_step,
                        const uint32_t* d_keepbits, polus_bf16_t* d_dqkv, float* d_gbias_qkv, void* stream);
/* d_gbias_qkv (may be NULL): [3*nh*head_dim] fp32, += column sums of d_dqkv -- the BiasAddGrad of the QKV projection
 * (polus/training.py:185), taken from the tiles while they are still in shared memory. */

/* dz = dy * act'(z); column sums of dz accumulated into d_gbias (bias gradient).
 * act == NONE with d_dz == NULL: bias gradient only.  d_ws: polus_colsum_ws_floats(N). */
int polus_act_bwd_colsum(const polus_bf16_t* d_dy, const polus_bf16_t* d_z, int M, int N, int act,
                         polus_bf16_t* d_dz, float* d_gbias, float* d_ws, void* stream);
size_t polus_colsum_ws_floats(int N);

/* tf.keras.layers.Dropout (polus/ner/models.py:58) on bf16 */
int polus_dropout(const polus_bf16_t* d_x, polus_bf16_t* d_y, int64_t n, float p_drop, uint64_t seed,
                  uint32_t site, const uint32_t* d_step, void* stream);

/* ---------------------------------------------------------------- CRF / losses -------------- */
/* tfa.text.crf_log_likelihood as used by polus/layers.py:86-126.  Per-sequence nll[b] =
 * log_norm - sequence_score; loss = mean_b(w[b]*nll[b]); gradients of that mean wrt emissions
 * [B,T,K] and transitions [K,K] (accumulated).  d_lens may be NULL (= T for all rows,
 * layers.py:74-76); d_weights may be NULL (= 1).  1 <= K <= 128; T up to the shared-memory limit of the
 * kernel that serves (K, T), at least 512 for every K. */
int polus_crf_nll(const float* d_emis, const int32_t* d_tags, const int32_t* d_lens,
                  const float* d_trans, const float* d_weights, int B, int T, int K,
                  float* d_nll, float* d_loss, float* d_gemis, float* d_gtrans, void* stream);
/* tfa.text.crf_decode (polus/layers.py:78-80): Viterbi, ties -> lowest index.  Same K and T limits. */
int polus_crf_decode(const float* d_emis, const int32_t* d_lens, const float* d_trans, int B, int T,
                     int K, int32_t* d_tags, float* d_score, void* stream);
/* CRF.get_transitions (polus/layers.py:56-63): T*mask + float(int32(1-mask)*-10000) */
int polus_crf_mask_transitions(const float* d_trans, const float* d_mask, int K, float* d_out,
                               void* stream);

/* CRF.loss_sample_weights (polus/layers.py:116-121): per-sequence weight from one-hot labels [B,T,K] */
int polus_crf_sample_weights(const float* d_y_true, const float* d_mask_positive, float negative_weight,
                             int B, int T, int K, float* d_out, void* stream);

/* kind 0: SparseCategoricalCrossentropy(from_logits) (tutorials/classifier_example.py:55), labels int32
 * kind 1: weighted softmax CE, one-hot/soft labels fp32 (polus/losses.py:5-18)
 * kind 2: weighted sigmoid CE, multi-hot labels fp32 (polus/losses.py:21-42)
 * loss = mean over rows; d_glogits = d loss / d logits. */
int polus_xent(int kind, const float* d_logits, const void* d_labels, const float* d_class_w,
               float negative_weight, int rows, int C, float* d_loss, float* d_glogits,
               void* stream);

/* ---------------------------------------------------------------- masked-language-model head  */
/* HF BertForMaskedLM / RobertaForMaskedLM at TF BERT's masked_lm_positions [B,P] (polus_version() >= 103).
 * Gather: d_out[b*P + j, :] = d_h[b, pos[b,j], :] over bf16 [B,S,H], H % 8 == 0; positions clamped to [0, S).
 * Scatter: d_dh[b, pos[b,j], :] += d_g[b*P + j, :]; a position named by several slots of a row receives their fp32 sum
 * (ascending j), rounded to bf16 once.  Deterministic; d_dh is normally zeroed by the caller.  P <= 12288 for the scatter. */
int polus_gather_positions(const polus_bf16_t* d_h, const int32_t* d_pos, int B, int S, int H, int P,
                           polus_bf16_t* d_out, void* stream);
int polus_scatter_positions_add(const polus_bf16_t* d_g, const int32_t* d_pos, int B, int S, int H, int P,
                                polus_bf16_t* d_dh, void* stream);
/* Cross-entropy over a vocabulary: bf16 logits [R,V], row stride ldl (>= V, multiple of 8), int32 labels [R] (clamped to
 * [0,V)), fp32 weights [R].  loss = sum_r w_r (lse_r - x_r[y_r]) / sum_r w_r, 0 when every weight is 0 (fp32 statistics).
 * Writes d_nll[r] = lse_r - x_r[y_r] and d_argmax[r] (lowest index on ties; may be NULL) and OVERWRITES the logits with
 * d loss / d logits (bf16; columns V..ldl untouched).  d_labels == NULL: inference, argmax only, logits untouched.
 * Any V >= 1, one code path. */
int polus_vocab_xent(polus_bf16_t* d_logits, int R, int V, int64_t ldl, const int32_t* d_labels, const float* d_weights,
                     float* d_nll, int32_t* d_argmax, float* d_loss, void* stream);
/* d_out[c] += sum_r d_x[r*ld + c], c < N (bias gradient of the vocabulary projection); one atomic per column per 64-row slab */
int polus_colsum_bf16(const polus_bf16_t* d_x, int R, int N, int64_t ld, float* d_out, void* stream);

/* ---------------------------------------------------------------- optimizer ----------------- */
typedef struct {
    float lr;            /* base LR (already multiplied by hvd.size(): training.py:90-94) */
    int32_t schedule;    /* 0 constant; 1 polus/schedulers.py:5-23 (linear warm-up + linear decay) */
    int32_t warmup_steps;
    int32_t decay_steps;
    float end_lr;        /* 1e-7 in the reference (schedulers.py:15) */
    float beta1, beta2, eps;
    float weight_decay;  /* 0: Keras Adam; >0: HF AdamWeightDecay (decoupled) */
    float grad_scale;    /* 1/world_size folded in (Horovod op=Average, training.py:182) */
} polus_adam_cfg_t;
/* Keras Adam over a flat arena: lr_t = lr*sqrt(1-b2^t)/(1-b1^t); p -= lr_t*m/(sqrt(v)+eps).
 * Also refreshes the bf16 shadow, zeroes g, and (thread 0) increments *d_step.
 * d_decay_mask: optional per-element u8 (1 = apply weight decay).
 * d_hyper: optional device float[4] {lr, grad_scale, weight_decay, end_lr} that overrides the same cfg
 * fields at run time -- cfg is frozen into a captured CUDA graph, the buffer is not, so
 * optimizer.learning_rate.assign() (training.py:90-94) takes effect on the next replay. */
int polus_adam(float* d_p, float* d_g, float* d_m, float* d_v, polus_bf16_t* d_p_bf16,
               const uint8_t* d_decay_mask, int64_t n, const polus_adam_cfg_t* cfg,
               const float* d_hyper, uint32_t* d_step, int increment_step, void* stream);

/* ---------------------------------------------------------------- small tensor utilities ---- */
int polus_cast(const void* d_src, int src_dtype, void* d_dst, int dst_dtype, int64_t n, void* stream);
int polus_fill_f32(float* d_dst, float value, int64_t n, void* stream);
/* op: 0 add, 1 sub, 2 mul, 3 div (fp32); b_n may be 1 (scalar broadcast) or == n or a row vector
 * of length `b_n` broadcast over rows (n % b_n == 0). */
int polus_binary_f32(int op, const float* d_a, const float* d_b, int64_t n, int64_t b_n,
                     float* d_out, void* stream);
/* op: polus_act_t codes 0..5, plus 16 exp, 17 log, 18 softplus, 19 sigmoid, 20 neg, 21 square,
 * 22 scale-by-alpha;
 * grad=1 computes dy * f'(x) into d_out (d_dy required). */
int polus_unary_f32(int op, const float* d_x, const float* d_dy, int grad, int64_t n, float* d_out,
                    float alpha, void* stream);
/* out[r] = sum_c x[r,c] (axis=1) or out[c] = sum_r x[r,c] (axis=0); scale applied. */
int polus_reduce_sum_f32(const float* d_x, int rows, int cols, int axis, float scale, float* d_out,
                         int accumulate, void* stream);
int polus_argmax_f32(const float* d_x, int rows, int cols, int32_t* d_out, void* stream);
int polus_one_hot_f32(const int32_t* d_idx, int rows, int cols, float* d_out, void* stream);
/* tf.math.confusion_matrix (polus/metrics.py:55-63): cm[true, pred] += 1 */
int polus_confusion_matrix(const int32_t* d_true, const int32_t* d_pred, int64_t n, int num_classes,
                           int32_t* d_cm, void* stream);
/* gather rows: out[i,:] = x[idx[i],:] (fp32/bf16 by elem_bytes); used for h[:,0,:] pooling */
int polus_gather_rows(const void* d_x, int64_t row_stride_bytes, int64_t row_bytes,
                      int64_t first_row, int64_t row_step, int64_t n_rows, void* d_out,
                      void* stream);
int polus_add_bf16(const polus_bf16_t* d_a, const polus_bf16_t* d_b, polus_bf16_t* d_out, int64_t n,
                   void* stream);
int polus_scatter_rows_add_bf16(const polus_bf16_t* d_g, int64_t cols, int64_t first_row,
                                int64_t row_step, int64_t n_rows, polus_bf16_t* d_out, void* stream);
/* global L2 norm (post_process_grads clipping, training.py:187-189) */
int polus_sumsq_f32(const float* d_x, int64_t n, float* d_out, void* stream);
int polus_scale_by_clip(float* d_x, int64_t n, const float* d_sumsq, float max_norm, void* stream);

/* ---------------------------------------------------------------- data-parallel comm -------- */
/* replaces horovod.tensorflow (polus/mock/horovod.py:5-24 is the surface; polus/training.py:182,
 * 208-211; polus/callbacks.py:249) with NCCL over NVLink. */
int polus_comm_unique_id(void* h_id128);            /* 128 bytes, call on rank 0 */
int polus_comm_init(int rank, int size, const void* h_id128);
/* same, capping the communicator's CTAs (ncclConfig_t.maxCTAs): the exchange runs under backward and every SM
 * NCCL holds is one the persistent GEMMs wait for; max_ctas <= 0 keeps NCCL's default */
int polus_comm_init_cfg(int rank, int size, const void* h_id128, int max_ctas);
int polus_comm_size(void);
int polus_comm_rank(void);
int polus_comm_allreduce_f32(float* d_buf, int64_t n, void* stream); /* sum, in place */
/* sum with a bf16 wire format: pack fp32 -> d_scratch (n bf16), ncclAllReduce(bf16), unpack into d_buf */
int polus_comm_allreduce_bf16(float* d_buf, polus_bf16_t* d_scratch, int64_t n, void* stream);
int polus_comm_broadcast(void* d_buf, size_t bytes, int root, void* stream);
int polus_comm_allgather(const void* d_send, void* d_recv, size_t bytes_per_rank, void* stream);
int polus_comm_destroy(void);

#ifdef __cplusplus
}
#endif
#endif /* POLUS_B200_H */
