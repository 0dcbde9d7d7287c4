/* libbdetr.so — C ABI of the B200-native Boosted_DETR hot path.
 *
 * The reference (mvenouziou/Boosted_DETR) has no FFI: its boundary is the Keras layer protocol
 * (pure Python).  Each entry point below replaces the body of one reference layer `call`; the
 * Python classes in boosted_detr_b200/ keep the reference's class names / ctor arguments / call
 * conventions and forward to these functions through ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C, no torch / CUDA-runtime types in signatures: device pointers are `void*`/`float*`,
 *     the stream is an opaque `void*` holding a cudaStream_t (NULL = legacy default stream);
 *   - every tensor is row-major fp32 in device memory unless stated otherwise; the caller owns all
 *     memory (inputs, outputs, saved activations, scratch); no hidden allocation, no hidden sync;
 *   - all calls are asynchronous on the given stream and CUDA-graph capturable;
 *   - return 0 (BDETR_OK) or a negative bdetr_status; bdetr_last_error() gives a thread-local text;
 *   - citations are file:line under /root/reference/ModelComponents/.
 */
#ifndef BDETR_H_
#define BDETR_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    BDETR_OK = 0,
    BDETR_E_BAD_SHAPE = -1,
    BDETR_E_CUDA = -2,
    BDETR_E_INVALID_COST = -3, /* scipy: ValueError("matrix contains invalid numeric entries") */
    BDETR_E_INFEASIBLE = -4,   /* scipy: ValueError("cost matrix is infeasible")               */
    BDETR_E_NULL = -5,
    BDETR_E_UNSUPPORTED = -6,
    BDETR_E_NCCL = -7          /* an NCCL call failed / libnccl could not be loaded (bdetr_last_error has the text) */
} bdetr_status;

/* compute modes for the dense (GEMM / attention) kernels */
#define BDETR_MODE_FP32 0 /* fp32 SIMT FFMA everywhere: the 1e-5 parity mode                   */
#define BDETR_MODE_TF32 1 /* TF32 operands (10-bit mantissa) via TMA, fp32 accumulate in TMEM on tcgen05 (1e-3 mode) */
#define BDETR_MODE_FP16 2 /* BDETR_MODE_TF32 with fp16 attention operands where the fp16 kernel serves the shape (long
                           * sequences: the config-5 encoder self-attention): q / k / v and the softmax weights P are fp16
                           * (tcgen05.mma kind::f16), accumulation fp32 -- the reference's Keras `mixed_float16` policy
                           * (parameters.py:73).  Needs bdetr_attn_saved.ws16 / the *_f16 entry point's workspace; shapes the
                           * fp16 kernel does not serve, and every backward, run exactly as in BDETR_MODE_TF32 (the Python
                           * layers hand ws16 over for inference forwards only). */

/* 101: attention at head dim 64 (D/H = 64) besides 32
 * 103: graph-captured inference with the early exit on the device (bdetr_exit_graph_*, bdetr_early_exit_decide)
 * 104: the attention core backward exported on its own (bdetr_attention_core_bwd)
 * 105: per-image early exit: images leave the batch at their own boundary (bdetr_image_exit_*, bdetr_switch_graph_*) */
int bdetr_version(void);
const char *bdetr_last_error(void);
/* Process-wide compute mode used by the dense entry points. */
int bdetr_set_mode(int mode);
int bdetr_get_mode(void);
/* Programmatic dependent launch (on by default): every kernel is launched with stream-serialisation relaxed and
 * blocks in griddepcontrol.wait before its first global access, so its prologue overlaps the previous kernel's
 * tail.  Semantics are unchanged (plain stream order); the switch exists for A/B timing. */
int bdetr_set_pdl(int on);
/* Intra-call concurrency (on by default): independent kernel chains inside one entry point (wgrad next to dgrad,
 * the q/k/v projections) run on library-owned auxiliary streams, forked from and joined back into the caller's
 * stream before the call returns; CUDA-graph capturable. */
int bdetr_set_concurrency(int on);
int bdetr_get_concurrency(void);
/* Deferred joins (off by default).  The fused backward entry points run their parameter-gradient side chains (weight
 * gradients, bias / positional gradients) on auxiliary streams.  With deferred joins on, an entry point returns without
 * ordering the caller's stream after those chains -- nothing inside the step reads parameter gradients -- and the
 * caller issues bdetr_join(stream) once, before it hands the gradients to the optimizer / all-reduce.  Data gradients
 * and everything the forward produces are always joined inside the call. */
int bdetr_set_deferred_join(int on);
int bdetr_join(void *stream);
/* the same, but `waiter` (e.g. the communication stream that all-reduces the gradients) is ordered after the chains that
 * were forked from `stream`, and `stream` itself keeps running */
int bdetr_join_into(void *stream, void *waiter);
int bdetr_get_pdl(void);
/* Number of kernels launched by this library since the last reset (bench.py's gpu_launches). */
long long bdetr_launch_count(void);
void bdetr_reset_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * Matcher trio (K7/K8/K9)
 * ---------------------------------------------------------------------------------------- */

/* Pairwise matching cost [B,T,Q] (targets = rows, predictions = columns):
 *   cost = (w_cat*cat + w_box*box) + w_attr*attr
 * Replaces CostArray.call (losses_and_metrics.py:222-225) applied to CategoryLoss (:44-49),
 * AttributeLoss (:51-57), BoxLoss (:68-72) plus the weighting / summation of MatchingLoss.call
 * (:119-130), without the reference's [B,T,Q,C] / [B,T,Q,A] / [B,T,Q,4] broadcast intermediates.
 * cat_true [B,T,C] one-hot, attr_true [B,T,A] multi-hot (entries must be exactly 0 or 1),
 * box_true [B,T,4], cat_pred [B,Q,C], attr_pred [B,Q,A], box_pred [B,Q,4] (COCO x,y,w,h). */
int bdetr_cost_matrix_fwd(int B, int T, int Q, int C, int A,
                          const float *cat_true, const float *attr_true, const float *box_true,
                          const float *cat_pred, const float *attr_pred, const float *box_pred,
                          float w_cat, float w_box, float w_attr,
                          float *cost, void *stream);

/* The same computation split in two, for callers that match the SAME targets against several prediction sets (the
 * boosted model: one target batch, N blocks) or that run matchers concurrently on several streams:
 *   bdetr_cost_targets_prepare  digests the target side once (class / attribute bit sets, class slots, hoisted box
 *                               invariants, padding-row detection) into `prepared`, a caller-owned device buffer of
 *                               bdetr_cost_targets_bytes(B,T,C,A) bytes, 16-byte aligned;
 *   bdetr_cost_matrix_prepared  builds cost[B,T,Q] from it; bit-identical to bdetr_cost_matrix_fwd.
 * bdetr_cost_matrix_fwd itself is these two calls on a library-owned grow-only scratch buffer (allocated on first use,
 * outside graph capture; one buffer per device, so not for concurrent use from several streams).
 * Limits (BDETR_E_UNSUPPORTED, before anything is launched):
 *   prepare   C <= 2048, A <= 1024, T*C and T*A < 2^22.  The target blocks are staged in shared memory when
 *             T*(C+A) floats plus the digest fit 227 KB and C <= 1024; otherwise they are read from global memory.
 *   cost      C <= 2048.  With Cs = C|1 and As = A|1, the cost tile takes
 *                 16 + 256*C (16-byte aligned) + digest + 256*Cs + attr + 256  bytes,
 *             digest = bdetr_cost_targets_bytes(1,T,C,A), attr = 0 when w_attr == 0, else 256*17 for A <= 4 and
 *             256*As above.  When that exceeds 227 KB the 256*C tile is dropped and 256*Cs becomes
 *             256*(min(C,T)|1) (the probabilities of the classes that occur are read from global memory); the call
 *             is refused if that still exceeds 227 KB, which only a large A can cause (A above about 620 at T = 100 and
 *             C = 2048, about 840 at T = 20 and C = 1205).
 *   Both paths give the same bits. */
size_t bdetr_cost_targets_bytes(int B, int T, int C, int A);
int bdetr_cost_targets_prepare(int B, int T, int C, int A,
                               const float *cat_true, const float *attr_true, const float *box_true,
                               void *prepared, void *stream);
int bdetr_cost_matrix_prepared(int B, int T, int Q, int C, int A, const void *prepared,
                               const float *cat_pred, const float *attr_pred, const float *box_pred,
                               float w_cat, float w_box, float w_attr,
                               float *cost, void *stream);

/* Per-image rectangular linear sum assignment on cost[b, :num_objects[b], :]; results are
 * bit-identical to scipy.optimize.linear_sum_assignment (ties included).
 * Replaces MatchingAssignment.scipy_linear_assignment_mask (:234-245) and MatchingMask.call
 * (:202-212).  Outputs (each may be NULL except col4row/status):
 *   col4row  [B,T] int32  matched prediction of target row t, -1 if none (padding / n>Q leftovers)
 *   row4col  [B,Q] int32  matched target of prediction q, -1 if none
 *   mask     [B,T,Q] fp32 the reference's assignment mask
 *   assigned [B,Q]   fp32 max_t mask (the reference's `assigned_predictions`)
 *   status   [B]   int32  0, BDETR_E_INVALID_COST or BDETR_E_INFEASIBLE per image (device flag;
 *                         the host wrapper polls it once per step, not per call). */
int bdetr_lsap_assign(int B, int T, int Q, const float *cost, const int32_t *num_objects,
                      int32_t *col4row, int32_t *row4col, float *mask, float *assigned,
                      int32_t *status, void *stream);
/* dynamic shared memory (bytes) one image needs in bdetr_lsap_assign; informational. */
size_t bdetr_lsap_smem_bytes(int T, int Q);

/* Matched losses of MatchingLoss.call (:133-160): losses [5,B] = total, category, attribute, box,
 * existence; iou [Q] = the `IOU` metric (shape [1,Q] in the reference, SURVEY quirk Q7).
 * weights = {w_cat, w_box, w_attr, w_exist}. */
int bdetr_matched_loss_fwd(int B, int T, int Q, int C, int A,
                           const float *cat_true, const float *attr_true, const float *box_true,
                           const int32_t *num_objects,
                           const float *cat_pred, const float *attr_pred, const float *box_pred,
                           const int32_t *col4row, const int32_t *row4col,
                           float w_cat, float w_box, float w_attr, float w_exist,
                           float *losses, float *iou, void *stream);

/* d(gscale * sum_b total_b)/d(predictions), ACCUMULATED (+=) into d_cat_pred [B,Q,C],
 * d_attr_pred [B,Q,A], d_box_pred [B,Q,4].  The assignment is a constant (tf.numpy_function). */
int bdetr_matched_loss_bwd(int B, int T, int Q, int C, int A,
                           const float *cat_true, const float *attr_true, const float *box_true,
                           const int32_t *num_objects,
                           const float *cat_pred, const float *attr_pred, const float *box_pred,
                           const int32_t *col4row, const int32_t *row4col,
                           float w_cat, float w_box, float w_attr, float w_exist, float gscale,
                           float *d_cat_pred, float *d_attr_pred, float *d_box_pred, void *stream);

/* MatchingMetric.call (:176-192): out [B,T,Q] = (mask ? mask : 1) * IoU(box_true[b,t], box_pred[b,q]) on COCO x,y,w,h boxes
 * (IOU_Metric :17-18).  mask may be NULL. */
int bdetr_pairwise_iou(int B, int T, int Q, const float *box_true, const float *box_pred, const float *mask, float *out,
                       void *stream);

/* Caller-owned buffers of the layer-level entry points, in bytes (no hidden allocation: the caller sizes `saved` /
 * `scratch` from these).  Each returns the total over the buffers of the corresponding struct, laid out as the struct's
 * comments state (fp32).  training = 0: what an inference call needs. */
size_t bdetr_attention_block_saved_bytes(int B, int Lq, int Lk, int D, int H, int training);
size_t bdetr_attention_block_scratch_bytes(int B, int Lq, int Lk, int D, int H);   /* bdetr_attn_scratch + d_resid + sums of the fused form */
size_t bdetr_ffn_block_saved_bytes(int M, int D, int training);
size_t bdetr_ffn_block_scratch_bytes(int M, int D);
size_t bdetr_heads_saved_bytes(int M, int Dh, int C, int A);
size_t bdetr_heads_scratch_bytes(int M, int Dh, int C, int A);

/* ------------------------------------------------------------------------------------------
 * Dense path (K1-K6)
 * ---------------------------------------------------------------------------------------- */

/* Keras Dense kernels are [in,out]; y = x @ kernel + bias. */
typedef struct {
    float *wq, *bq, *wk, *bk, *wv, *bv, *wo, *bo; /* [D,D] / [D] each                   */
    float *ln_gamma, *ln_beta;                   /* [D]                                 */
} bdetr_attn_params;                             /* same struct is used for gradients   */

/* caller-allocated activations saved by the forward for the backward (also forward scratch) */
typedef struct {
    float *qp, *kp, *vp; /* projected q [B,Lq,D], k,v [B,Lk,D]                              */
    float *o;            /* attention output in the reference's [B,H,Lq,d] layout (quirk Q1) */
    float *lse;          /* [B,H,Lq] log-sum-exp of the scaled scores                        */
    float *z;            /* [B,Lq,D] pre-LayerNorm sum                                       */
    float *mean, *rstd;  /* [B*Lq] LayerNorm statistics                                      */
    void *ws16;          /* BDETR_MODE_FP16 only (else NULL): bdetr_attention_f16_workspace_bytes() bytes, 128-byte
                          * aligned, for the fp16 copies of qp / kp / vp; NULL keeps the TF32 kernel        */
} bdetr_attn_saved;

/* backward scratch: d_qp [B,Lq,D], d_kp, d_vp [B,Lk,D], d_o [B,H,Lq,d], d_z [B,Lq,D], delta [B,H,Lq] */
typedef struct {
    float *d_qp, *d_kp, *d_vp, *d_o, *d_z, *delta;
} bdetr_attn_scratch;

/* AttentionBlock.call (transformers.py:139-151) with MultiheadAttention.call (:68-102) inside:
 *   out = LayerNorm_eps( query + Dropout( MHA(query,key,value) ) )
 * query [B,Lq,D] (also the residual), key/value [B,Lk,D]; H heads of width D/H, which must be 32 or 64 (other widths
 * return BDETR_E_UNSUPPORTED); the attention output is re-read as [B,Lq,D] WITHOUT permuting back (reference line :100).
 * dropout_rate 0 disables dropout (inference); the keep mask is hash(idx ^ key) >= rate * 2^32 with
 * key = dropout_key when dropout_seed_dev is NULL, else key = lowbias32(*dropout_seed_dev ^ dropout_key): the
 * per-step seed is then read from DEVICE memory by the kernels, so a captured CUDA graph draws a fresh mask on every
 * replay (Keras Dropout semantics, reference transformers.py:135,147) once the caller refreshes that word. */
int bdetr_attention_block_fwd(int B, int Lq, int Lk, int D, int H,
                              const float *query, const float *key, const float *value,
                              const bdetr_attn_params *w, float dropout_rate, uint32_t dropout_key,
                              const uint32_t *dropout_seed_dev, float ln_eps, float *out,
                              const bdetr_attn_saved *saved, void *stream);

/* The attention core alone (transformers.py:77-97): qp [B,Lq,H*d], kp/vp [B,Lk,H*d] are the projected tensors
 * (head = d-column slice), o [B,H,Lq,d], lse [B,H,Lq] (log2 units); d = 32 or 64.  Scores are never written to HBM.
 * Tensor-core mode runs the tcgen05/TMEM flash kernel; fp32 mode the SIMT kernel. */
int bdetr_attention_core_fwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                             float *o, float *lse, void *stream);
/* Backward of bdetr_attention_core_fwd: qp [B,Lq,H*d], kp/vp [B,Lk,H*d], o / d_o [B,H,Lq,d], lse [B,H,Lq] (log2 units,
 * as the forward writes it); writes delta [B,H,Lq] = sum_d d_o*o, d_qp [B,Lq,H*d], d_kp / d_vp [B,Lk,H*d] (overwritten,
 * not rounded).  Tensor-core mode: the tcgen05 kernels; fp32 mode: the SIMT kernels.  d = 32 or 64. */
int bdetr_attention_core_bwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                             const float *o, const float *lse, const float *d_o, float *delta,
                             float *d_qp, float *d_kp, float *d_vp, void *stream);

/* fp16-operand attention core (BDETR_MODE_FP16; reference policy: parameters.py:73 `mixed_float16`).  Same contract as
 * bdetr_attention_core_fwd; ws16 = bdetr_attention_f16_workspace_bytes(...) bytes of caller-owned scratch (fp16 copies of
 * qp / kp / vp).  The workspace query returns 0 for shapes the fp16 kernel does not serve (it needs head dim 32, Lq >= 1536,
 * Lk >= 1024 and at least 148 CTAs of 384 query rows); the entry point then returns BDETR_E_UNSUPPORTED. */
size_t bdetr_attention_f16_workspace_bytes(int B, int H, int Lq, int Lk, int d);
int bdetr_attention_core_fwd_f16(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                                 void *ws16, float *o, float *lse, void *stream);

/* Backward of the above.  Parameter gradients are ACCUMULATED into *gw.  d_query/d_key/d_value
 * may be NULL (not needed); acc_flags bit0/1/2 = accumulate into d_query/d_key/d_value instead of
 * overwriting. */
int bdetr_attention_block_bwd(int B, int Lq, int Lk, int D, int H,
                              const float *query, const float *key, const float *value,
                              const bdetr_attn_params *w, float dropout_rate, uint32_t dropout_key,
                              const uint32_t *dropout_seed_dev, const bdetr_attn_saved *saved, const float *d_out,
                              float *d_query, float *d_key, float *d_value, int acc_flags,
                              const bdetr_attn_params *gw, const bdetr_attn_scratch *scratch,
                              void *stream);

typedef struct {
    float *w1, *b1, *w2, *b2; /* DenseRelu, DenseLinear: [D,D] / [D] */
    float *ln_gamma, *ln_beta;
} bdetr_ffn_params;

typedef struct {
    float *h;           /* [M,D] relu(x W1 + b1)        */
    float *z;           /* [M,D] pre-LayerNorm sum      */
    float *mean, *rstd; /* [M]                          */
} bdetr_ffn_saved;

typedef struct {
    float *d_z, *d_h; /* [M,D] each */
} bdetr_ffn_scratch;

/* FeedForwardBlock.call (transformers.py:182-193): out = LN( x + Dropout( relu(xW1+b1)W2+b2 ) ). */
int bdetr_ffn_block_fwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                        float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                        float *out, const bdetr_ffn_saved *saved, void *stream);
int bdetr_ffn_block_bwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                        float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                        const bdetr_ffn_saved *saved, const float *d_out,
                        float *d_x, int accumulate_dx,
                        const bdetr_ffn_params *gw, const bdetr_ffn_scratch *scratch, void *stream);

/* out[b,l,:] = x[b,l,:] + pos[l,:]  (EncoderBlock Add1/Add2 :226-227, DecoderPrep Add :441). */
int bdetr_add_positional_fwd(int B, int L, int D, const float *x, const float *pos, float *out,
                             void *stream);
/* d_pos[l,:] += sum_b d_out[b,l,:]. */
int bdetr_add_positional_bwd(int B, int L, int D, const float *d_out, float *d_pos, void *stream);
/* out[b,q,:] = q0[q,:]  (DecoderPrep TileBatch2D :445-447) and its backward d_q0 += sum_b d_out. */
int bdetr_tile_queries_fwd(int B, int Q, int D, const float *q0, float *out, void *stream);
/* y += x elementwise (gradient joins). */
int bdetr_accumulate(size_t n, const float *x, float *y, void *stream);
/* buf [n,len]: buf[i] += buf[i+1] for i = n-2 .. 0.  The boosted running prediction of block i feeds the losses of blocks
 * i .. n-1 (boosted_model.py:222-246), so its gradient is the suffix sum of the per-block loss gradients. */
int bdetr_suffix_sum(int n, size_t len, float *buf, void *stream);
/* dst = round-to-nearest tf32(src) (may alias).  Tensor-core mode keeps tf32-rounded shadows of the Dense
 * kernels and of the input features so that tcgen05's operand truncation is exact. */
int bdetr_round_tf32(size_t n, const float *src, float *dst, void *stream);

/* One prediction head = Dense(relu) -> BatchNorm -> Dense -> activation, post-activation output
 * added into the running (boosted) prediction:  cum += mult * act(...), mult = 2 for block 0
 * (boosted_model.py:222-229, quirk Q2).
 * kind: 0 softmax (SingleClassPredictionHead, prediction_heads.py:113-131)
 *       1 sigmoid (MultiClassPredictionHead :182-201)
 *       2 3*sigmoid(x/100)-1 (BoxPredictionHead :46-63) */
typedef struct {
    float *w1, *b1;                  /* [D,Dh], [Dh]                           */
    float *bn_gamma, *bn_beta;       /* [Dh]                                   */
    float *bn_moving_mean, *bn_moving_var; /* [Dh] (updated in training)       */
    float *w2, *b2;                  /* [Dh,Nout], [Nout]                      */
} bdetr_head_params;

typedef struct {
    float *h;                /* [M,Dh] relu(x W1 + b1)               */
    float *hn;               /* [M,Dh] batch-normalised              */
    float *bn_mean, *bn_rstd;/* [Dh]                                 */
    float *bn_acc;           /* [2*Dh*ceil(M/128)] scratch for the per-row-chunk column sums */
    float *act;              /* [M,Nout] post-activation output      */
} bdetr_head_saved;

typedef struct {
    float *d_logits; /* [M,Nout] */
    float *d_hn;     /* [M,Dh]   */
    float *d_h;      /* [M,Dh]   */
} bdetr_head_scratch;

int bdetr_head_fwd(int M, int D, int Dh, int Nout, int kind, int training, float mult,
                   const float *x, const bdetr_head_params *w, float bn_eps, float bn_momentum,
                   float *cum, int cum_init, const bdetr_head_saved *saved, void *stream);
/* d_cum [M,Nout] is the gradient w.r.t. the running prediction this head was added into.  bn_training must equal the
 * `training` flag of the forward call: 0 = the BatchNorm used its moving statistics (inference, or a frozen head -- a
 * non-trainable Keras BatchNormalization runs in inference mode), so they are constants in the backward. */
int bdetr_head_bwd(int M, int D, int Dh, int Nout, int kind, int bn_training, float mult,
                   const float *x, const bdetr_head_params *w, float bn_eps,
                   const bdetr_head_saved *saved, const float *d_cum,
                   float *d_x, int accumulate_dx,
                   const bdetr_head_params *gw, const bdetr_head_scratch *scratch, void *stream);

/* ------------------------------------------------------------------------------------------
 * Fused tensor-core path (tcgen05 / TMEM / TMA, tf32 operands, fp32 accumulation) -- what the model runs in
 * BDETR_MODE_TF32.  These entry points ARE the tensor-core path (they do not consult bdetr_set_mode): every tensor that
 * feeds a GEMM must already be rounded to tf32 by its producer (bdetr_round_tf32 for inputs / weight shadows; the kernels
 * round what they produce).  Same math as the layer-level entry points above, in fewer, fatter kernels:
 *   - q / k / v projections: ONE grouped GEMM; the positional add of EncoderBlock (:226-227) / DecoderPrep (:441) is
 *     folded in as a batch-invariant row table, (x + pos) W + b = x W + (pos W + b)   [bdetr_pos_projection];
 *   - output projection / DenseLinear + bias + Dropout + residual (+ pos rows, quirk Q4) + LayerNorm: ONE kernel whose
 *     CTA owns whole 256-wide rows (reference :101,147-149 / :187-191);
 *   - backward: one grouped weight-gradient GEMM and one k-concatenated data-gradient GEMM per projection group, bias
 *     gradients from the epilogues / the batch-reduction kernel, positional gradients from batch-summed rows.
 * NULL gradient outputs skip work: gw == NULL (frozen block: no parameter gradients), d_* == NULL (nothing trainable
 * upstream) -- the reference's per-block freezing schedule (Boosted_DETR_COCO.ipynb cell 30).
 * ---------------------------------------------------------------------------------------- */

/* tab[g] [L,D] = pos_tc [L,D] @ W[g] [D,D] + b[g] [D]   for g < n <= 3: one grouped GEMM, once per step and block
 * (batch-invariant).  pos_tc / W: tf32-rounded copies. */
int bdetr_pos_projection(int L, int D, const float *pos_tc, int n, const float *const *W, const float *const *b,
                         float *const *tab, void *stream);

typedef struct {
    const float *pos;     /* [L,D] positional table (L = Lk; = Lq too when resid_pos / tab_q are used, else BDETR_E_BAD_SHAPE); NULL: none */
    const float *tab_q;   /* [Lq,D] pos Wq + bq, or NULL: q = query Wq + bq                                         */
    const float *tab_k;   /* [Lk,D] pos Wk + bk, or NULL: k = key Wk + bk                                           */
    int resid_pos;        /* 1: the residual is query + pos (encoder, quirk Q4: transformers.py:148 with :226)      */
    const float *pos_tc;  /* tf32-rounded copy of pos: tensor-core operand of the backward's positional GEMMs        */
} bdetr_pos_fold;

/* AttentionBlock.call with the positional adds folded in.  query [B,Lq,D]; memory [B,Lk,D] is the input of BOTH the key
 * and the value projection (encoder: memory == query == x, k = (x+pos) Wk; decoder: memory = encoder output).
 * saved->z may be NULL when training == 0 (nothing is kept for a backward).  */
int bdetr_attention_fused_fwd(int B, int Lq, int Lk, int D, int H, const float *query, const float *memory,
                              const bdetr_pos_fold *fold, const bdetr_attn_params *w,
                              float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                              int training, float *out, const bdetr_attn_saved *saved, void *stream);

/* scratch: bdetr_attn_scratch as above plus
 *   d_resid [B,Lq,D]  gradient of the residual input (query + pos)
 *   sums    [4,max(Lq,Lk),D]  batch sums (residual, d_qp, d_kp, spare)
 * d_query [B,Lq,D] (NULL: skipped) receives residual + q-path (+ k/v paths when memory == query);
 * d_memory [B,Lk,D] (NULL or ignored when memory == query) the k/v paths; acc flags bit0 / bit1 accumulate instead of
 * overwriting.  d_pos [L,D] is accumulated (NULL: skipped). */
int bdetr_attention_fused_bwd(int B, int Lq, int Lk, int D, int H, const float *query, const float *memory,
                              const bdetr_pos_fold *fold, const bdetr_attn_params *w,
                              float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                              const bdetr_attn_saved *saved, const float *d_out,
                              float *d_query, float *d_memory, int acc_flags, float *d_pos,
                              const bdetr_attn_params *gw, const bdetr_attn_scratch *scratch, float *d_resid, float *sums,
                              void *stream);

/* FeedForwardBlock.call: DenseRelu as one GEMM, DenseLinear + Dropout + residual + LayerNorm as one kernel. */
int bdetr_ffn_fused_fwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                        float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                        int training, float *out, const bdetr_ffn_saved *saved, void *stream);
int bdetr_ffn_fused_bwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                        float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                        const bdetr_ffn_saved *saved, const float *d_out, float *d_x, int accumulate_dx,
                        const bdetr_ffn_params *gw, const bdetr_ffn_scratch *scratch, void *stream);

/* Decoder self-attention block (DecoderBlock.call :378-380: q = k = v = the shared queries, no positional term), hoisted
 * out of the batch: the projections, the attention core and the output projection depend on the [Q,D] query parameter
 * only and run ONCE per step ([1,Q,D]); only Dropout + residual + LayerNorm run per image.
 *   q0 [Q,D] (q0_tc: its tf32-rounded copy, the GEMM operand); out [B,Q,D]; saved: qp,kp,vp [Q,D], o [H,Q,d], lse [H,Q], z [B,Q,D], mean,rstd [B*Q]; mha [Q,D] = the
 *   attention output before Dropout. */
int bdetr_decoder_self_fwd(int B, int Q, int D, int H, const float *q0, const float *q0_tc, const bdetr_attn_params *w,
                           float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                           int training, float *out, const bdetr_attn_saved *saved, float *mha, void *stream);
/* d_q0 [Q,D] accumulated.  scratch: d_qp,d_kp,d_vp [Q,D], d_o [H,Q,d], delta [H,Q], d_z [B,Q,D]; d_resid [B,Q,D];
 * sums [2,Q,D]. */
int bdetr_decoder_self_bwd(int B, int Q, int D, int H, const float *q0, const float *q0_tc, const bdetr_attn_params *w,
                           float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                           const bdetr_attn_saved *saved, const float *d_out, float *d_q0,
                           const bdetr_attn_params *gw, const bdetr_attn_scratch *scratch, float *d_resid, float *sums,
                           void *stream);

/* The three prediction heads of one boosted block in one call (prediction_heads.py:46-63,113-131,182-201 +
 * boosted_model.py:222-229):  hidden layers as ONE grouped GEMM, BatchNorm folded into the second Dense
 * ((h - mu) * rstd * gamma + beta) W2 + b2 = h (diag(rstd*gamma) W2) + ((beta - mu*rstd*gamma) W2 + b2), second Dense +
 * activation + boosted running sum in one fp32 kernel: cum_out[k] = (cum_in[k] ? cum_in[k] : 0) + mult * act_k(...).
 * heads[0..2] = category (softmax, Nout = C), attribute (sigmoid, A), box (3*sigmoid(x/100)-1, 4).
 *   saved: h [3,M,Dh] post-ReLU hidden activations, bn_mean / bn_rstd [3,Dh], w2f / b2f [3,Dh] the affine map
 *   hn = h * w2f + b2f the output kernel folds into the second Dense, bn_part scratch, act[k] [M,Nout_k] post-activation
 *   outputs.  C, A <= 2048 (BDETR_E_UNSUPPORTED above, before anything is launched).  A head of more than 320
 *   outputs computes its logits in column slabs of 320 and then runs the row activation and the running sum as a
 *   second kernel; narrower heads run the one-kernel path.
 * bn_training[k] = 0: head k normalises with its moving statistics (inference, or a frozen head). */
typedef struct {
    float *h, *bn_mean, *bn_rstd, *w2f, *b2f;
    float *bn_part;    /* [ceil(M/128), 2, 3*Dh] scratch: per-row-chunk column sums (deterministic BatchNorm statistics) */
    float *act[3];
} bdetr_heads_saved;
typedef struct {
    float *d_logits;   /* [M, C+A+4]                                         */
    float *hTd;        /* [3*Dh*max(C,A,4)] h^T d_logits per head (+ colsums) */
    float *colsum_d;   /* [C+A+4]                                            */
    float *bn_s;       /* [2,3,Dh] batch-norm backward sums                  */
    float *d_h;        /* [3,M,Dh]                                           */
} bdetr_heads_scratch;
int bdetr_heads_fwd(int M, int D, int Dh, int C, int A, const float *x, const bdetr_head_params *heads /* [3] */,
                    const int *bn_training /* [3] */, float bn_eps, float bn_momentum, float mult,
                    const float *const *cum_in /* [3], entries may be NULL */, float *const *cum_out /* [3] */,
                    const bdetr_heads_saved *saved, void *stream);
/* d_cum[k] [M,Nout_k]: gradient w.r.t. the running prediction.  gw[k] == NULL skips head k's parameter gradients
 * (frozen); d_x NULL skips the input gradient. */
int bdetr_heads_bwd(int M, int D, int Dh, int C, int A, const float *x, const bdetr_head_params *heads,
                    const int *bn_training, float mult, const bdetr_heads_saved *saved, const float *const *d_cum,
                    float *d_x, int accumulate_dx, const bdetr_head_params *const *gw /* [3] */,
                    const bdetr_heads_scratch *scratch, void *stream);

/* Debug aid: when non-NULL, CTA (0,0,0) of every tcgen05 GEMM writes eight clock64 stamps into this device
 * buffer (entry, setup done, 2nd TMA issue, first stage landed, last MMA committed, accumulator ready,
 * epilogue done, teardown).  Pass NULL to switch it off. */
int bdetr_debug_set_timeline(long long *device_buf8);
/* Debug / test aid: which tcgen05 attention-forward kernel the tensor-core mode uses.  0 = automatic (multi-stream
 * kernel for long sequences, one tile per CTA otherwise), 1 = always one tile per CTA, 2 = always multi-stream;
 * 20 + n = multi-stream with n of every 8 exponential groups evaluated on the FMA pipe.  The multi-stream kernel serves
 * head dim 32 only: at head dim 64 the automatic choice is the one-tile kernel, and forcing 2 or 20 + n makes the
 * attention forward return BDETR_E_UNSUPPORTED without launching anything. */
int bdetr_debug_force_attention_kernel(int which);

/* Generic row-major GEMM used by the entry points above, exported for tests and benchmarks:
 * C[M,N] = (beta ? C : 0) + op(A)[M,K] @ op(B)[K,N] (+ bias[N]) (relu if act==1).
 * transA: A is stored [K,M]; transB: B is stored [N,K]. */
int bdetr_gemm(int M, int N, int K, const float *A, int transA, const float *Bm, int transB,
               const float *bias, int act, int beta, float *C, void *stream);

/* ------------------------------------------------------------------------------------------
 * Optimizer step (SURVEY 8f rank 1): Keras SGD with momentum / Nesterov and per-variable clipnorm, the optimizer of
 * the reference's training runs (Boosted_DETR_COCO.ipynb cells 26, 30:
 * tf.keras.optimizers.SGD(learning_rate=lr, momentum=.9, nesterov=True, clipnorm=0.1)).
 *   g <- (g * clipnorm) / max(||g||_2, clipnorm) per variable  (tf.clip_by_norm; clipnorm <= 0 disables it)
 *   accum <- momentum * accum - lr * g ;  var += nesterov ? momentum * accum - lr * g : accum
 * The trainable variables are described by a DEVICE table of chunks (<= 16384 elements each, a variable = a run of
 * consecutive table entries) over the flat weight / gradient / accumulator buffers; frozen variables are simply left
 * out of the table.  `partial` = n_chunks floats of workspace.  The schedule (CosineDecayRestarts, ...) is evaluated by
 * the host side; the step's learning rate is the plain argument `lr`, or -- when `lr_dev` is not NULL -- the float it
 * points to in device memory (so that a captured CUDA graph can be replayed with a new rate every step).
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    long long offset;     /* first element of the chunk in the flat buffers */
    int len;              /* elements in the chunk */
    int var_first;        /* table index of the first chunk of the variable this chunk belongs to */
    int var_chunks;       /* number of chunks of that variable */
    int reserved;
} bdetr_opt_chunk;

int bdetr_sgd_step(int n_chunks, const bdetr_opt_chunk *chunks,
                   float *weights, const float *grads, float *accum, float *partial,
                   float lr, const float *lr_dev, float momentum, int nesterov, float clipnorm, void *stream);

/* ------------------------------------------------------------------------------------------
 * BackboneNeck (SURVEY 8f rank 2; reference backbone.py:66-95): BatchNorm -> 1x1 Conv2D(Cin -> N, tanh) -> BatchNorm on
 * the channels-last backbone feature map, M = B*rows*cols pixels.  One tcgen05 GEMM with BN1 folded into the weights,
 * tanh in the epilogue, BN2 as one affine pass (round_out: stored tf32-rounded, ready to be block 0's operand).
 * x_tc [M,Cin]: the backbone output rounded to tf32 (bdetr_round_tf32).  Keras BatchNormalization: momentum .99, eps 1e-3.
 *   saved: t [M,N] tanh output, wf [Cin,N] / bf [N] folded weights, part scratch of max(ceil(M/128)*2*Cin, ceil(Cin/32)*N) floats,
 *          stat1 [4,Cin] / stat2 [4,N] = mean, rstd, scale, shift of the two normalisations.
 * Backward: parameter gradients only (the backbone is frozen in the reference, notebook cell 30); scratch d_u [M,N],
 * gwf [Cin*N + N].
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    float *bn1_gamma, *bn1_beta, *bn1_moving_mean, *bn1_moving_var;   /* [Cin] */
    float *conv_w, *conv_b;                                           /* [Cin,N] (the [1,1,Cin,N] Conv2D kernel), [N] */
    float *bn2_gamma, *bn2_beta, *bn2_moving_mean, *bn2_moving_var;   /* [N] */
} bdetr_neck_params;
typedef struct {
    float *t, *wf, *bf, *part, *stat1, *stat2;
} bdetr_neck_saved;
int bdetr_backbone_neck_fwd(int M, int Cin, int N, const float *x_tc, const bdetr_neck_params *w, float bn_eps, float bn_momentum,
                            int training, float *out, const bdetr_neck_saved *saved, int round_out, void *stream);
int bdetr_backbone_neck_bwd(int M, int Cin, int N, const float *x_tc, const bdetr_neck_params *w, int training,
                            const bdetr_neck_saved *saved, const float *d_out, const bdetr_neck_params *gw, float *d_u, float *gwf,
                            void *stream);

/* ------------------------------------------------------------------------------------------
 * Inference tail (SURVEY 8f rank 3): the numeric half of InverseTokenization.call (tokenizers.py:126-137) and the
 * confidence statistic of the early-exit path the reference lists as TODO (README.md:9).
 *   tokens_categories [B,Q] int32 = argmax_c cat_pred (first maximum, like tf.argmax)
 *   tokens_attributes [B,Q,A] int32 = (attr_pred >= .5) * arange(A)
 *   confidence [B,Q] = conf_scale * max_c cat_pred ; image_confidence [B] = min_q confidence
 * Any output may be NULL (image_confidence needs confidence).  conf_scale = 1 / (number of summed softmax vectors).
 * ---------------------------------------------------------------------------------------- */
int bdetr_inverse_tokenize(int B, int Q, int C, int A, const float *cat_pred, const float *attr_pred,
                           int32_t *tokens_categories, int32_t *tokens_attributes, float *confidence,
                           float *image_confidence, float conf_scale, void *stream);

/* ------------------------------------------------------------------------------------------
 * Graph-captured inference with the early exit decided on the device (conditional graph nodes, CUDA 12.4+).
 * A forward of N boosted blocks has N - 1 boundaries; boundary i decides whether block i + 1 runs.  The caller
 *   1. bdetr_exit_graph_create(N - 1, &g, handles): the top-level graph and one IF-node handle per boundary;
 *   2. captures N + 1 segments on its own: S0 = everything before block 0 plus block 0, Sk = block k (k >= 1),
 *      E = bdetr_select_exit_predictions.  Each Sk with k < N - 1 ends with bdetr_inverse_tokenize of block k's running
 *      category prediction and bdetr_early_exit_decide(boundary k, next_block = handles[k]).  A segment must not wait on
 *      an event recorded in another one, and may contain kernel, memset, memcpy, empty and child-graph nodes only (the
 *      nodes CUDA allows inside a conditional body);
 *   3. bdetr_exit_graph_build(g, segments, N + 1) -> child(S0) -> IF(h0){S1} -> ... -> IF(h_{N-2}){S_{N-1}} -> child(E),
 *      instantiated (the segments are cloned: the caller may destroy its own graphs afterwards);
 *   4. bdetr_exit_graph_launch(g, stream) per call; bdetr_exit_graph_destroy(g) at the end.
 * Every handle resets to 0 at launch, so once a boundary exits, no later block runs.
 * ---------------------------------------------------------------------------------------- */
#define BDETR_MAX_EXIT_BLOCKS 32
typedef struct bdetr_exit_graph bdetr_exit_graph;
int bdetr_exit_graph_create(int n_boundaries, bdetr_exit_graph **g, unsigned long long *handles);
int bdetr_exit_graph_build(bdetr_exit_graph *g, void *const *segments, int n_segments);
int bdetr_exit_graph_launch(bdetr_exit_graph *g, void *stream);
int bdetr_exit_graph_destroy(bdetr_exit_graph *g);
/* One CTA.  image_conf [B] = the image confidences of the running prediction after block `boundary` (bdetr_inverse_tokenize
 * with conf_scale = 1 / (boundary + 2)).  Device words: threshold (float32), min_blocks, threshold_set (0 / 1).  Block
 * boundary + 1 runs when boundary + 1 < min_blocks, or threshold_set == 0, or some image has !(image_conf >= threshold)
 * (the eager rule: float32 compare, inclusive, a NaN confidence is not confident).  Writes exit_block = boundary when it
 * exits and n_blocks - 1 otherwise, copies image_conf into conf_out [B], and sets the condition of `next_block` (0 = no
 * conditional node: the decision is only written). */
int bdetr_early_exit_decide(int B, int boundary, int n_blocks, const float *image_conf, const float *threshold,
                            const int32_t *min_blocks, const int32_t *threshold_set, unsigned long long next_block,
                            int32_t *exit_block, float *conf_out, void *stream);
/* cums [3 * n_blocks] = the running category [B,Q,C], attribute [B,Q,A] and box [B,Q,4] predictions of block 0, 1, ...;
 * copies those of block *exit_block (read on the device) into cat / attr / box.  n_blocks <= BDETR_MAX_EXIT_BLOCKS. */
int bdetr_select_exit_predictions(int n_blocks, int B, int Q, int C, int A, const float *const *cums,
                                  const int32_t *exit_block, float *cat, float *attr, float *box, void *stream);

/* ------------------------------------------------------------------------------------------
 * Per-image early exit (inference).  Each image leaves the forward after its own boundary; the images still running are
 * gathered to the front of the batch in order and the next block runs at that smaller batch k.  On a path whose GEMMs need
 * k_min rows' worth of images (the fused tensor-core path: k_min = max(ceil(128 / L), ceil(128 / Q))) the batch never
 * drops below k_min: images that have already left ride along (recomputed, never written again).
 *   state   int32 words, bdetr_image_exit_state_bytes(B, N) bytes, allocated by the caller; nothing needs initialising.
 *           word 0 n_active (images running the next block, riders included), 1 .. N counts[N] (images that ran each block),
 *           then exit_block[B] (int32), conf[B] (float32: the image's confidence at its exit boundary, or at the last
 *           boundary checked; NaN if none was), then private words (the slot order, the gather list, per-slot flags).
 *   after block i < N - 1, on the block's stream:
 *     bdetr_inverse_tokenize(k_in, ...) of the k_in running slots' category prediction, conf_scale = 1 / (i + 2);
 *     bdetr_image_exit_plan(.., boundary i, k_in, image_conf, threshold, min_blocks, threshold_set, switch handle | 0, state):
 *       one CTA; image_conf [k_in] in slot order; device words as for bdetr_early_exit_decide.  A live image leaves when
 *       threshold_set, i + 1 >= min_blocks and image_conf >= threshold (float32, a NaN is not confident).  Writes the
 *       new slot order and n_active = 0 if nobody stays, else max(stayers, k_min).  With a handle, sets it to
 *       n_active - k_min, or B - k_min + 1 (no body) when nobody stays.  k_in == B at boundary 0.
 *     bdetr_image_exit_compact(.., boundary i, k_in, ..): the running predictions cum_in [3] ([k_in, Q, C | A | 4]) of the
 *       images leaving here -> out [3] ([B, Q, .]) at their original index; x_in [k_in, x_row] and cum_in of the next
 *       block's slots -> x_out / cum_out (separate buffers of B rows; n_active rows are written, read on the device).
 *   after block N - 1: bdetr_image_exit_compact(.., boundary N - 1, ..) writes every live slot's predictions to out
 *     (x_in, x_out, cum_out may be NULL).  Needs n_blocks >= 2.
 * ---------------------------------------------------------------------------------------- */
size_t bdetr_image_exit_state_bytes(int B, int n_blocks);
int bdetr_image_exit_plan(int B, int n_blocks, int k_min, int boundary, int k_in, const float *image_conf,
                          const float *threshold, const int32_t *min_blocks, const int32_t *threshold_set,
                          unsigned long long next_switch, int32_t *state, void *stream);
int bdetr_image_exit_compact(int B, int n_blocks, int boundary, int k_in, int Q, int C, int A, long long x_row,
                             const float *x_in, const float *const *cum_in, float *x_out, float *const *cum_out,
                             float *const *out, const int32_t *state, void *stream);
/* Graph of the per-image exit (SWITCH nodes, CUDA 12.8 driver or newer, else BDETR_E_UNSUPPORTED):
 *   bdetr_switch_graph_create(N - 1, n_branches = B - k_min + 1, &g, handles): one SWITCH handle per boundary, default
 *     value n_branches (matches no body: a SWITCH whose plan did not run launches nothing);
 *   capture S0 = everything before block 0 + block 0 + boundary 0's plan (handle 0) and compaction, and for every
 *     boundary i = 0 .. N - 2 and k = k_min .. B the body S_{i+1}@k = block i + 1 at batch k + boundary i + 1's plan
 *     (handle i + 1) and compaction, or the final compaction in block N - 1;
 *   bdetr_switch_graph_build(g, {S0, S1@k_min .. S1@B, S2@k_min, ...}, 1 + (N - 1) * n_branches)
 *     -> child(S0) -> SWITCH(h0){S1@k_min .. S1@B} -> ... -> SWITCH(h_{N-2}){S_{N-1}@k_min .. S_{N-1}@B};
 *   bdetr_exit_graph_launch / bdetr_exit_graph_destroy as above. */
int bdetr_switch_graph_create(int n_boundaries, int n_branches, bdetr_exit_graph **g, unsigned long long *handles);
int bdetr_switch_graph_build(bdetr_exit_graph *g, void *const *segments, int n_segments);

/* ------------------------------------------------------------------------------------------
 * Data parallel (SURVEY 8e): the gradient all-reduce, the only collective on the path.  The reference's
 * tf.distribute.MirroredStrategy (parameters.py:74) sums the replica gradients with TF-internal NCCL; here one NCCL
 * communicator per device lives behind an opaque bdetr_comm (libnccl bound at run time with dlopen).
 *   rank 0:      bdetr_comm_unique_id(id)  -> hand the 128 bytes to every rank by any out-of-band channel
 *   every rank:  cudaSetDevice(local) ; bdetr_comm_init(&comm, rank, world, id)
 *   per step:    bdetr_allreduce(comm, flat_grads + lo, hi - lo, stream)   in-place sum, stream-ordered, graph capturable
 * ---------------------------------------------------------------------------------------- */
typedef struct bdetr_comm bdetr_comm;
int bdetr_comm_unique_id(void *id128);
int bdetr_comm_init(bdetr_comm **comm, int rank, int world, const void *id128);
int bdetr_comm_destroy(bdetr_comm *comm);
int bdetr_comm_info(const bdetr_comm *comm, int *rank, int *world, int *nccl_version);
int bdetr_allreduce(bdetr_comm *comm, float *buf, size_t count, void *stream);
int bdetr_broadcast(bdetr_comm *comm, float *buf, size_t count, int root, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* BDETR_H_ */
