// C-ABI entry points of the dense path: each one replaces the body of one reference Keras layer
// `call` and is a short sequence of kernel launches on the caller's stream (no allocation, no sync).
#include "kernels.cuh"

using namespace bdetr;
#define API extern "C" __attribute__((visibility("default")))
#define TRY(x) do { int rc__ = (x); if (rc__ != BDETR_OK) return rc__; } while (0)

// Tensor-core mode: every tensor that feeds a tcgen05 GEMM is stored rounded to tf32 (round-to-nearest) by
// its producer, so the MMA's operand truncation is exact.  `rnd` below is that flag.
static inline int tc_mode() { return current_mode() == BDETR_MODE_TF32 ? 1 : 0; }

// y = x @ W + b, W is a Keras kernel [K,N]
static int linear_fwd(int M, int N, int K, const float *x, const float *W, const float *b, int act, float *y, int rnd, cudaStream_t s)
{
    return launch_gemm(M, N, K, x, K, false, W, N, false, b, act, nullptr, 0, rnd, y, N, s);
}
// Backward of y = x W + b, as two independent halves (they run on different streams, see Branches):
// weight half: gW += x^T dy ; gb += colsum(dy)
static int linear_wgrad(int M, int N, int K, const float *x, const float *dy, float *gW, float *gb, cudaStream_t s)
{
    if (gW) TRY(launch_gemm(K, N, M, x, K, true, dy, N, false, nullptr, 0, nullptr, 1, 0, gW, N, s));
    if (gb) TRY(launch_colsum_acc(M, N, dy, gb, s));
    return BDETR_OK;
}
// data half: dx (=|+=) dy W^T (optionally masked by relu_mask afterwards)
static int linear_dgrad(int M, int N, int K, const float *W, const float *dy, float *dx, int acc_dx, const float *relu_mask,
                        int rnd_dx, cudaStream_t s)
{
    return launch_gemm(M, K, N, dy, N, false, W, N, true, nullptr, 0, relu_mask, acc_dx, rnd_dx, dx, K, s);
}

API int bdetr_gemm(int M, int N, int K, const float *A, int transA, const float *Bm, int transB,
                   const float *bias, int act, int beta, float *C, void *stream)
{
    return launch_gemm(M, N, K, A, transA ? M : K, transA != 0, Bm, transB ? K : N, transB != 0, bias, act, nullptr,
                       beta, 0, C, N, as_stream(stream));
}

API int bdetr_attention_block_fwd(int B, int Lq, int Lk, int D, int H,
                                  const float *query, const float *key, const float *value,
                                  const bdetr_attn_params *w, float dropout_rate, uint32_t dropout_key,
                                  const uint32_t *dropout_seed_dev, float ln_eps, float *out, const bdetr_attn_saved *sv, void *stream)
{
    BDETR_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && D > 0 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(query && key && value && w && out && sv, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(sv->qp && sv->kp && sv->vp && sv->o && sv->lse && sv->z && sv->mean && sv->rstd, BDETR_E_NULL, "null saved buffer");
    cudaStream_t s = as_stream(stream);
    const int Mq = B * Lq, Mk = B * Lk;
    const int rnd = tc_mode();
    // q/k/v feed the tcgen05 attention MMAs in tensor-core mode: store them tf32-rounded
    Branches br(s);
    cudaStream_t sk = br.fork(0), sv_s = br.fork(1);          // the three projections are independent
    TRY(linear_fwd(Mq, D, D, query, w->wq, w->bq, 0, sv->qp, rnd, s));
    TRY(linear_fwd(Mk, D, D, key, w->wk, w->bk, 0, sv->kp, rnd, sk));
    TRY(linear_fwd(Mk, D, D, value, w->wv, w->bv, 0, sv->vp, rnd, sv_s));
    TRY(br.join());
    TRY(launch_attention_fwd(B, H, Lq, Lk, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, rnd, s));
    // sv->o is [B,H,Lq,d]; read back as [B*Lq, D] with no permute (reference transformers.py:100)
    TRY(linear_fwd(Mq, D, D, sv->o, w->wo, w->bo, 0, sv->z, 0, s));
    TRY(launch_res_ln_fwd(Mq, D, query, sv->z, w->ln_gamma, w->ln_beta, ln_eps, dropout_rate, dropout_key, dropout_seed_dev, out, sv->mean, sv->rstd, rnd, s));
    return BDETR_OK;
}

API int bdetr_attention_core_fwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                                 float *o, float *lse, void *stream)
{
    BDETR_REQUIRE(qp && kp && vp && o && lse, BDETR_E_NULL, "null pointer");
    return launch_attention_fwd(B, H, Lq, Lk, d, qp, kp, vp, o, lse, 0, as_stream(stream));
}

API int bdetr_attention_core_bwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                                 const float *o, const float *lse, const float *d_o, float *delta,
                                 float *d_qp, float *d_kp, float *d_vp, void *stream)
{
    BDETR_REQUIRE(qp && kp && vp && o && lse && d_o && delta && d_qp && d_kp && d_vp, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(B > 0 && H > 0 && Lq > 0 && Lk > 0, BDETR_E_BAD_SHAPE, "bad attention shape");
    return launch_attention_bwd(B, H, Lq, Lk, d, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, 0, as_stream(stream));
}

API size_t bdetr_attention_f16_workspace_bytes(int B, int H, int Lq, int Lk, int d)
{
    if (B <= 0 || H <= 0 || Lq <= 0 || Lk <= 0) return 0;
    return attention_f16_workspace_bytes(B, H, Lq, Lk, d);
}

API int bdetr_attention_core_fwd_f16(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                                     void *ws16, float *o, float *lse, void *stream)
{
    BDETR_REQUIRE(qp && kp && vp && o && lse && ws16, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(B > 0 && H > 0 && Lq > 0 && Lk > 0, BDETR_E_BAD_SHAPE, "bad attention shape");
    BDETR_REQUIRE(attention_f16_workspace_bytes(B, H, Lq, Lk, d) > 0, BDETR_E_UNSUPPORTED, "shape not served by the fp16 attention kernel");
    return launch_attention_fwd_umma_ms_f16(B, H, Lq, Lk, d, qp, kp, vp, ws16, o, lse, 0, as_stream(stream));
}

API int bdetr_attention_block_bwd(int B, int Lq, int Lk, int D, int H,
                                  const float *query, const float *key, const float *value,
                                  const bdetr_attn_params *w, float dropout_rate, uint32_t dropout_key,
                                  const uint32_t *dropout_seed_dev, const bdetr_attn_saved *sv, const float *d_out,
                                  float *d_query, float *d_key, float *d_value, int acc_flags,
                                  const bdetr_attn_params *gw, const bdetr_attn_scratch *sc, void *stream)
{
    BDETR_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && D > 0 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(query && key && value && w && sv && d_out && gw && sc, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(sc->d_qp && sc->d_kp && sc->d_vp && sc->d_o && sc->d_z && sc->delta, BDETR_E_NULL, "null scratch buffer");
    cudaStream_t s = as_stream(stream);
    const int Mq = B * Lq, Mk = B * Lk;
    // LayerNorm + residual + dropout: residual gradient goes straight to d_query
    const int rnd = tc_mode();
    TRY(launch_res_ln_bwd(Mq, D, d_out, sv->z, sv->mean, sv->rstd, w->ln_gamma, dropout_rate, dropout_key, dropout_seed_dev,
                          d_query, acc_flags & 1, sc->d_z, gw->ln_gamma, gw->ln_beta, gw->bo, rnd, s));
    // output projection (its bias gradient was fused into the LayerNorm backward above): the weight half runs
    // beside the data path.  d_o feeds the tcgen05 attention backward MMAs in tensor-core mode: stored tf32-rounded
    Branches br(s);
    TRY(linear_wgrad(Mq, D, D, sv->o, sc->d_z, gw->wo, nullptr, br.fork(0)));
    TRY(linear_dgrad(Mq, D, D, w->wo, sc->d_z, sc->d_o, 0, nullptr, rnd, s));
    TRY(launch_attention_bwd(B, H, Lq, Lk, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, sc->d_o, sc->delta,
                             sc->d_qp, sc->d_kp, sc->d_vp, rnd, s));
    // the three weight halves on three auxiliary streams; the data halves stay in order on the caller's stream
    // because d_query / d_key / d_value may alias (q = k in the encoder, q = k = v in decoder self-attention)
    TRY(linear_wgrad(Mq, D, D, query, sc->d_qp, gw->wq, gw->bq, br.fork(0)));
    TRY(linear_wgrad(Mk, D, D, key, sc->d_kp, gw->wk, gw->bk, br.fork(1)));
    TRY(linear_wgrad(Mk, D, D, value, sc->d_vp, gw->wv, gw->bv, br.fork(2)));
    TRY(linear_dgrad(Mq, D, D, w->wq, sc->d_qp, d_query, 1, nullptr, 0, s));
    TRY(linear_dgrad(Mk, D, D, w->wk, sc->d_kp, d_key, (acc_flags >> 1) & 1, nullptr, 0, s));
    TRY(linear_dgrad(Mk, D, D, w->wv, sc->d_vp, d_value, (acc_flags >> 2) & 1, nullptr, 0, s));
    return br.join();
}

API int bdetr_ffn_block_fwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                            float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                            float *out, const bdetr_ffn_saved *sv, void *stream)
{
    BDETR_REQUIRE(M > 0 && D > 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(x && w && out && sv && sv->h && sv->z && sv->mean && sv->rstd, BDETR_E_NULL, "null pointer");
    cudaStream_t s = as_stream(stream);
    const int rnd = tc_mode();
    TRY(linear_fwd(M, D, D, x, w->w1, w->b1, 1, sv->h, rnd, s));
    TRY(linear_fwd(M, D, D, sv->h, w->w2, w->b2, 0, sv->z, 0, s));
    TRY(launch_res_ln_fwd(M, D, x, sv->z, w->ln_gamma, w->ln_beta, ln_eps, dropout_rate, dropout_key, dropout_seed_dev, out, sv->mean, sv->rstd, rnd, s));
    return BDETR_OK;
}

API int bdetr_ffn_block_bwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                            float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                            const bdetr_ffn_saved *sv, const float *d_out,
                            float *d_x, int accumulate_dx,
                            const bdetr_ffn_params *gw, const bdetr_ffn_scratch *sc, void *stream)
{
    BDETR_REQUIRE(M > 0 && D > 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(x && w && sv && d_out && d_x && gw && sc && sc->d_z && sc->d_h, BDETR_E_NULL, "null pointer");
    cudaStream_t s = as_stream(stream);
    const int rnd = tc_mode();
    TRY(launch_res_ln_bwd(M, D, d_out, sv->z, sv->mean, sv->rstd, w->ln_gamma, dropout_rate, dropout_key, dropout_seed_dev,
                          d_x, accumulate_dx, sc->d_z, gw->ln_gamma, gw->ln_beta, gw->b2, rnd, s));
    // DenseLinear (bias gradient fused above), then ReLU mask on the way into DenseRelu; weight halves run beside
    Branches br(s);
    TRY(linear_wgrad(M, D, D, sv->h, sc->d_z, gw->w2, nullptr, br.fork(0)));
    TRY(linear_dgrad(M, D, D, w->w2, sc->d_z, sc->d_h, 0, sv->h, rnd, s));
    TRY(linear_wgrad(M, D, D, x, sc->d_h, gw->w1, gw->b1, br.fork(1)));
    TRY(linear_dgrad(M, D, D, w->w1, sc->d_h, d_x, 1, nullptr, 0, s));
    return br.join();
}

API int bdetr_add_positional_fwd(int B, int L, int D, const float *x, const float *pos, float *out, void *stream)
{
    BDETR_REQUIRE(x && pos && out, BDETR_E_NULL, "null pointer");
    return launch_add_rows_fwd(B, L, D, x, pos, out, tc_mode(), as_stream(stream));
}
API int bdetr_add_positional_bwd(int B, int L, int D, const float *d_out, float *d_pos, void *stream)
{
    BDETR_REQUIRE(d_out && d_pos, BDETR_E_NULL, "null pointer");
    return launch_batch_sum_acc(B, L, D, d_out, d_pos, as_stream(stream));
}
API int bdetr_tile_queries_fwd(int B, int Q, int D, const float *q0, float *out, void *stream)
{
    BDETR_REQUIRE(q0 && out, BDETR_E_NULL, "null pointer");
    return launch_tile_rows(B, Q, D, q0, out, tc_mode(), as_stream(stream));
}
API int bdetr_accumulate(size_t n, const float *x, float *y, void *stream)
{
    return launch_accumulate(n, x, y, as_stream(stream));
}
API int bdetr_suffix_sum(int n, size_t len, float *buf, void *stream)
{
    return launch_suffix_sum(n, len, buf, as_stream(stream));
}
API int bdetr_debug_force_attention_kernel(int which)
{
    BDETR_REQUIRE((which >= 0 && which <= 2) || (which >= 20 && which <= 28), BDETR_E_UNSUPPORTED,
                  "0 auto, 1 one tile per CTA, 2 multi-stream, 20 + n multi-stream with n of 8 exponential groups on the FMA pipe");
    bdetr::g_force_attention_kernel = which;
    return BDETR_OK;
}
namespace bdetr { extern long long *g_umma_timeline; }
API int bdetr_debug_set_timeline(long long *device_buf8)
{
    bdetr::g_umma_timeline = device_buf8;
    return BDETR_OK;
}
API int bdetr_round_tf32(size_t n, const float *src, float *dst, void *stream)
{
    return launch_round_tf32(n, src, dst, as_stream(stream));
}

API int bdetr_head_fwd(int M, int D, int Dh, int Nout, int kind, int training, float mult,
                       const float *x, const bdetr_head_params *w, float bn_eps, float bn_momentum,
                       float *cum, int cum_init, const bdetr_head_saved *sv, void *stream)
{
    BDETR_REQUIRE(M > 0 && D > 0 && Dh > 0 && Nout > 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(x && w && cum && sv && sv->h && sv->hn && sv->bn_mean && sv->bn_rstd && sv->bn_acc && sv->act, BDETR_E_NULL, "null pointer");
    cudaStream_t s = as_stream(stream);
    TRY(linear_fwd(M, Dh, D, x, w->w1, w->b1, 1, sv->h, 0, s));
    TRY(launch_bn_fwd(M, Dh, sv->h, w->bn_gamma, w->bn_beta, w->bn_moving_mean, w->bn_moving_var, bn_eps, bn_momentum,
                      training, sv->bn_acc, sv->hn, sv->bn_mean, sv->bn_rstd, s));
    TRY(linear_fwd(M, Nout, Dh, sv->hn, w->w2, w->b2, 0, sv->act, 0, s));
    TRY(launch_head_act_fwd(M, Nout, kind, mult, sv->act, cum, cum_init, s));
    return BDETR_OK;
}

API int bdetr_head_bwd(int M, int D, int Dh, int Nout, int kind, int bn_training, float mult,
                       const float *x, const bdetr_head_params *w, float bn_eps,
                       const bdetr_head_saved *sv, const float *d_cum,
                       float *d_x, int accumulate_dx,
                       const bdetr_head_params *gw, const bdetr_head_scratch *sc, void *stream)
{
    (void)bn_eps;
    BDETR_REQUIRE(M > 0 && D > 0 && Dh > 0 && Nout > 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(x && w && sv && d_cum && d_x && gw && sc && sc->d_logits && sc->d_hn && sc->d_h, BDETR_E_NULL, "null pointer");
    cudaStream_t s = as_stream(stream);
    TRY(launch_head_act_bwd(M, Nout, kind, mult, sv->act, d_cum, sc->d_logits, s));
    Branches br(s);
    TRY(linear_wgrad(M, Nout, Dh, sv->hn, sc->d_logits, gw->w2, gw->b2, br.fork(0)));
    TRY(linear_dgrad(M, Nout, Dh, w->w2, sc->d_logits, sc->d_hn, 0, nullptr, 0, s));
    TRY(launch_bn_relu_bwd(M, Dh, sv->h, sc->d_hn, w->bn_gamma, sv->bn_mean, sv->bn_rstd, sv->bn_acc, sc->d_h, gw->bn_gamma,
                           gw->bn_beta, gw->b1, tc_mode(), bn_training, s));
    TRY(linear_wgrad(M, Dh, D, x, sc->d_h, gw->w1, nullptr, br.fork(1)));
    TRY(linear_dgrad(M, Dh, D, w->w1, sc->d_h, d_x, accumulate_dx, nullptr, 0, s));
    return br.join();
}
