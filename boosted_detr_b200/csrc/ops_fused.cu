// Fused tensor-core path (include/bdetr.h "Fused tensor-core path"): the same layers as ops.cu in fewer, fatter
// kernels -- grouped q/k/v projection with the positional add folded in as a row table, Dense + Dropout + residual +
// LayerNorm in one tcgen05 kernel, grouped weight-gradient GEMMs, k-concatenated data-gradient GEMMs, one batch-reduction
// kernel for the bias / positional gradients, and the batch-invariant decoder self-attention hoisted out of the batch.
#include "kernels.cuh"

using namespace bdetr;
#define API extern "C" __attribute__((visibility("default")))
#define TRY(x) do { int rc__ = (x); if (rc__ != BDETR_OK) return rc__; } while (0)

namespace {

struct Proj {       // one Dense of a projection group
    const float *W, *b; float *out;
};

// out[g] = A @ W[g] (+ b[g]) (+ tab[g][row % period]) for up to 3 projections of ONE input; stored tf32-rounded
int proj_group_fwd(int M, int D, const float *A, int n, const Proj *p, const float *const *tab, int period, cudaStream_t s)
{
    GroupedGemm g;
    g.M = M; g.N = D; g.K = D; g.groups = n; g.share_a = true; g.lda = g.ldb = g.ldc = D; g.round_out = 1;
    g.A[0] = A;
    for (int i = 0; i < n; ++i) {
        g.B[i] = p[i].W; g.C[i] = p[i].out;
        g.bias[i] = tab[i] ? nullptr : p[i].b;          // the table already holds pos W + b
        g.rowtab[i] = tab[i];
    }
    g.rowtab_period = period; g.rowtab_ld = D;
    return launch_gemm_umma_grouped(g, s);
}

// gW[g] += A^T dY[g]  (A [M,D] shared, dY[g] [M,D]): grouped weight gradient, split-K atomics
int proj_group_wgrad(int M, int D, const float *A, int n, const float *const *dY, float *const *gW, cudaStream_t s)
{
    GroupedGemm g;
    g.M = D; g.N = D; g.K = M; g.groups = n; g.share_a = true; g.TA = true; g.lda = g.ldb = g.ldc = D; g.beta = 1;
    g.A[0] = A;
    for (int i = 0; i < n; ++i) { g.B[i] = dY[i]; g.C[i] = gW[i]; }
    return launch_gemm_umma_grouped(g, s);
}

// dX (=|+=) addend + sum_g dY[g] W[g]^T : ONE GEMM whose k loop runs over the groups
int proj_group_dgrad(int M, int D, int n, const float *const *dY, const float *const *W, const float *addend, int addend_period,
                     float *dX, int acc, cudaStream_t s)
{
    GroupedGemm g;
    g.M = M; g.N = D; g.K = D; g.groups = n; g.sum_groups = true; g.TB = true; g.lda = g.ldb = g.ldc = D; g.beta = acc;
    for (int i = 0; i < n; ++i) { g.A[i] = dY[i]; g.B[i] = W[i]; }
    g.C[0] = dX;
    g.rowtab[0] = addend; g.rowtab_period = addend_period; g.rowtab_ld = D;
    return launch_gemm_umma_grouped(g, s);
}

inline bool tc_rows_ok(long long M) { return M >= 1; }

// The fold's pos / pos_tc / d_pos have L = Lk rows (include/bdetr.h).  The residual reads pos[row % Lq] and the q path's
// positional gradient runs over Lq rows, so resid_pos and tab_q need Lq == Lk.
inline bool fold_rows_ok(const bdetr_pos_fold *fold, int Lq, int Lk)
{
    return !fold || Lq == Lk || !(fold->resid_pos || fold->tab_q);
}

}  // namespace

API int bdetr_pos_projection(int L, int D, const float *pos_tc, int n, const float *const *W, const float *const *b,
                             float *const *tab, void *stream)
{
    BDETR_REQUIRE(L > 0 && D > 0 && n >= 1 && n <= 3, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(pos_tc && W && b && tab, BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    GroupedGemm g;
    g.M = L; g.N = D; g.K = D; g.groups = n; g.share_a = true; g.lda = g.ldb = g.ldc = D;
    g.A[0] = pos_tc;
    for (int i = 0; i < n; ++i) { g.B[i] = W[i]; g.bias[i] = b[i]; g.C[i] = tab[i]; }
    return launch_gemm_umma_grouped(g, as_stream(stream));
}

API int bdetr_attention_fused_fwd(int B, int Lq, int Lk, int D, int H, const float *query, const float *memory,
                                  const bdetr_pos_fold *fold, const bdetr_attn_params *w,
                                  float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                                  int training, float *out, const bdetr_attn_saved *sv, void *stream)
{
    BDETR_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && D == 256 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "fused attention block needs D = 256");
    BDETR_REQUIRE(query && memory && w && out && sv, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(sv->qp && sv->kp && sv->vp && sv->o && sv->lse && sv->mean && sv->rstd && (sv->z || !training), BDETR_E_NULL, "null saved buffer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const int Mq = B * Lq, Mk = B * Lk;
    const float *tab_q = fold ? fold->tab_q : nullptr, *tab_k = fold ? fold->tab_k : nullptr;
    const float *rpos = (fold && fold->resid_pos) ? fold->pos : nullptr;
    BDETR_REQUIRE(!(fold && fold->resid_pos) || fold->pos, BDETR_E_NULL, "resid_pos needs the positional table");
    BDETR_REQUIRE(fold_rows_ok(fold, Lq, Lk), BDETR_E_BAD_SHAPE, "resid_pos / tab_q need Lq == Lk (pos has Lk rows)");
    const bool self = memory == query && Lq == Lk;
    if (self) {
        const Proj p[3] = {{w->wq, w->bq, sv->qp}, {w->wk, w->bk, sv->kp}, {w->wv, w->bv, sv->vp}};
        const float *tab[3] = {tab_q, tab_k, nullptr};
        TRY(proj_group_fwd(Mq, D, query, 3, p, tab, Lq, s));
    } else {
        Branches br(s);
        const Proj pq[1] = {{w->wq, w->bq, sv->qp}};
        const float *tq[1] = {tab_q};
        TRY(proj_group_fwd(Mq, D, query, 1, pq, tq, Lq, br.fork(0)));
        const Proj pkv[2] = {{w->wk, w->bk, sv->kp}, {w->wv, w->bv, sv->vp}};
        const float *tkv[2] = {tab_k, nullptr};
        TRY(proj_group_fwd(Mk, D, memory, 2, pkv, tkv, Lk, s));
        TRY(br.join());
    }
    if (attention_f16_enabled() && sv->ws16 && attention_f16_workspace_bytes(B, H, Lq, Lk, D / H) > 0)
        TRY(launch_attention_fwd_umma_ms_f16(B, H, Lq, Lk, D / H, sv->qp, sv->kp, sv->vp, sv->ws16, sv->o, sv->lse, 1, s));
    else
        TRY(launch_attention_fwd(B, H, Lq, Lk, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, 1, s));
    // sv->o is [B,H,Lq,d], read back as [B*Lq, D] with no permute (reference transformers.py:100, quirk Q1)
    TRY(launch_gemm_ln(Mq, D, sv->o, w->wo, w->bo, query, rpos, Lq, w->ln_gamma, w->ln_beta, ln_eps, dropout_rate, dropout_key,
                       dropout_seed_dev, training ? sv->z : nullptr, out, sv->mean, sv->rstd, 1, s));
    return BDETR_OK;
}

API int bdetr_attention_fused_bwd(int B, int Lq, int Lk, int D, int H, const float *query, const float *memory,
                                  const bdetr_pos_fold *fold, const bdetr_attn_params *w,
                                  float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                                  const bdetr_attn_saved *sv, const float *d_out,
                                  float *d_query, float *d_memory, int acc_flags, float *d_pos,
                                  const bdetr_attn_params *gw, const bdetr_attn_scratch *sc, float *d_resid, float *sums,
                                  void *stream)
{
    BDETR_REQUIRE(B > 0 && Lq > 0 && Lk > 0 && D == 256 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "fused attention block needs D = 256");
    BDETR_REQUIRE(query && memory && w && sv && d_out && sc && d_resid, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(sc->d_qp && sc->d_kp && sc->d_vp && sc->d_o && sc->d_z && sc->delta, BDETR_E_NULL, "null scratch buffer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const int Mq = B * Lq, Mk = B * Lk;
    const bool self = memory == query && Lq == Lk;
    const float *tab_q = fold ? fold->tab_q : nullptr, *tab_k = fold ? fold->tab_k : nullptr;
    const bool resid_pos = fold && fold->resid_pos;
    const float *pos_tc = fold ? (fold->pos_tc ? fold->pos_tc : fold->pos) : nullptr;
    const bool want_pos = d_pos != nullptr && (tab_q || tab_k || resid_pos);
    BDETR_REQUIRE(fold_rows_ok(fold, Lq, Lk), BDETR_E_BAD_SHAPE, "resid_pos / tab_q need Lq == Lk (pos has Lk rows)");
    BDETR_REQUIRE(!want_pos || (sums && pos_tc), BDETR_E_NULL, "positional gradients need `sums` and the positional table");
    const bool need_dq = d_query != nullptr, need_dm = !self && d_memory != nullptr;
    // LayerNorm + residual + dropout; the residual gradient lands in d_resid, the output projection's bias gradient is
    // the column sum of d_z
    TRY(launch_res_ln_bwd(Mq, D, d_out, sv->z, sv->mean, sv->rstd, w->ln_gamma, dropout_rate, dropout_key, dropout_seed_dev,
                          d_resid, 0, sc->d_z, gw ? gw->ln_gamma : nullptr, gw ? gw->ln_beta : nullptr, gw ? gw->bo : nullptr, 1, s));
    Branches br(s);
    if (gw) TRY(launch_gemm(D, D, Mq, sv->o, D, true, sc->d_z, D, false, nullptr, 0, nullptr, 1, 0, gw->wo, D, br.fork(0)));
    TRY(launch_gemm(Mq, D, D, sc->d_z, D, false, w->wo, D, true, nullptr, 0, nullptr, 0, 1, sc->d_o, D, s));
    TRY(launch_attention_bwd(B, H, Lq, Lk, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, sc->d_o, sc->delta,
                             sc->d_qp, sc->d_kp, sc->d_vp, 1, s));
    // ---- side chain: batch sums -> bias gradients, positional gradients --------------------------------------------
    if (gw || want_pos) {
        cudaStream_t ss = br.fork(1);
        BatchReduce r;
        r.B = B; r.D = D;
        float *S_r = sums, *S_q = sums ? sums + (size_t)Lq * D : nullptr, *S_k = sums ? sums + (size_t)Lq * D + (size_t)Lq * D : nullptr;
        auto add = [&](const float *src, int rows, float *sum, float *colsum) {
            if (!sum && !colsum) return;
            r.src[r.n] = src; r.rows[r.n] = rows; r.sum[r.n] = sum; r.colsum[r.n] = colsum; ++r.n;
        };
        add(d_resid, Lq, (want_pos && resid_pos) ? S_r : nullptr, nullptr);
        add(sc->d_qp, Lq, ((want_pos || gw) && tab_q) ? S_q : nullptr, gw ? gw->bq : nullptr);
        add(sc->d_kp, Lk, ((want_pos || gw) && tab_k) ? S_k : nullptr, gw ? gw->bk : nullptr);
        add(sc->d_vp, Lk, nullptr, gw ? gw->bv : nullptr);
        if (r.n) TRY(launch_batch_reduce(r, ss));
        if (want_pos && (tab_q || tab_k)) {
            // d_pos += R + S_q Wq^T + S_k Wk^T
            const float *dY[2]; const float *Wm[2]; int n = 0;
            if (tab_q) { dY[n] = S_q; Wm[n] = w->wq; ++n; }
            if (tab_k) { dY[n] = S_k; Wm[n] = w->wk; ++n; }
            TRY(proj_group_dgrad(tab_q ? Lq : Lk, D, n, dY, Wm, resid_pos ? S_r : nullptr, Lq, d_pos, 1, ss));
        } else if (want_pos && resid_pos) {
            TRY(launch_accumulate((size_t)Lq * D, S_r, d_pos, ss));
        }
        if (gw && (tab_q || tab_k)) {
            // gW[q|k] += pos^T S[q|k]   (the positional half of (x + pos)^T dY)
            const float *dY[2]; float *gW[2]; int n = 0;
            if (tab_q) { dY[n] = S_q; gW[n] = gw->wq; ++n; }
            if (tab_k) { dY[n] = S_k; gW[n] = gw->wk; ++n; }
            TRY(proj_group_wgrad(tab_q ? Lq : Lk, D, pos_tc, n, dY, gW, ss));
        }
    }
    // ---- weight gradients beside the data gradients ----------------------------------------------------------------
    if (self) {
        if (gw) {
            const float *dY[3] = {sc->d_qp, sc->d_kp, sc->d_vp}; float *gW[3] = {gw->wq, gw->wk, gw->wv};
            TRY(proj_group_wgrad(Mq, D, query, 3, dY, gW, br.fork(2)));
        }
        if (need_dq) {
            const float *dY[3] = {sc->d_qp, sc->d_kp, sc->d_vp}; const float *Wm[3] = {w->wq, w->wk, w->wv};
            TRY(proj_group_dgrad(Mq, D, 3, dY, Wm, d_resid, Mq, d_query, acc_flags & 1, s));
        }
    } else {
        if (gw) {
            const float *dYq[1] = {sc->d_qp}; float *gWq[1] = {gw->wq};
            TRY(proj_group_wgrad(Mq, D, query, 1, dYq, gWq, br.fork(2)));
            const float *dY[2] = {sc->d_kp, sc->d_vp}; float *gW[2] = {gw->wk, gw->wv};
            TRY(proj_group_wgrad(Mk, D, memory, 2, dY, gW, br.fork(0)));
        }
        if (need_dq) {
            const float *dY[1] = {sc->d_qp}; const float *Wm[1] = {w->wq};
            TRY(proj_group_dgrad(Mq, D, 1, dY, Wm, d_resid, Mq, d_query, acc_flags & 1, s));
        }
        if (need_dm) {
            const float *dY[2] = {sc->d_kp, sc->d_vp}; const float *Wm[2] = {w->wk, w->wv};
            TRY(proj_group_dgrad(Mk, D, 2, dY, Wm, nullptr, Mk, d_memory, (acc_flags >> 1) & 1, s));
        }
    }
    return br.join_deferrable();
}

API int bdetr_ffn_fused_fwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                            float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                            int training, float *out, const bdetr_ffn_saved *sv, void *stream)
{
    BDETR_REQUIRE(M > 0 && D == 256, BDETR_E_BAD_SHAPE, "fused FFN block needs D = 256");
    BDETR_REQUIRE(x && w && out && sv && sv->h && sv->mean && sv->rstd && (sv->z || !training), BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    GroupedGemm g;
    g.M = M; g.N = D; g.K = D; g.lda = g.ldb = g.ldc = D; g.round_out = 1; g.act = 1;
    g.A[0] = x; g.B[0] = w->w1; g.bias[0] = w->b1; g.C[0] = sv->h;
    TRY(launch_gemm_umma_grouped(g, s));
    TRY(launch_gemm_ln(M, D, sv->h, w->w2, w->b2, x, nullptr, 1, w->ln_gamma, w->ln_beta, ln_eps, dropout_rate, dropout_key,
                       dropout_seed_dev, training ? sv->z : nullptr, out, sv->mean, sv->rstd, 1, s));
    return BDETR_OK;
}

API int bdetr_ffn_fused_bwd(int M, int D, const float *x, const bdetr_ffn_params *w,
                            float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                            const bdetr_ffn_saved *sv, const float *d_out, float *d_x, int accumulate_dx,
                            const bdetr_ffn_params *gw, const bdetr_ffn_scratch *sc, void *stream)
{
    BDETR_REQUIRE(M > 0 && D == 256, BDETR_E_BAD_SHAPE, "fused FFN block needs D = 256");
    BDETR_REQUIRE(x && w && sv && d_out && d_x && sc && sc->d_z && sc->d_h, BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    TRY(launch_res_ln_bwd(M, D, d_out, sv->z, sv->mean, sv->rstd, w->ln_gamma, dropout_rate, dropout_key, dropout_seed_dev,
                          d_x, accumulate_dx, sc->d_z, gw ? gw->ln_gamma : nullptr, gw ? gw->ln_beta : nullptr, gw ? gw->b2 : nullptr, 1, s));
    Branches br(s);
    // d_h = (d_z W2^T) masked by relu'(h); its column sums are DenseRelu's bias gradient (epilogue)
    GroupedGemm g;
    g.M = M; g.N = D; g.K = D; g.TB = true; g.lda = g.ldb = g.ldc = D; g.round_out = 1; g.relu_mask = sv->h;
    g.A[0] = sc->d_z; g.B[0] = w->w2; g.C[0] = sc->d_h; g.colsum[0] = gw ? gw->b1 : nullptr;
    TRY(launch_gemm_umma_grouped(g, s));
    if (gw) {
        // both weight gradients in ONE grouped split-K launch on a side chain: gW2 += h^T d_z, gW1 += x^T d_h
        GroupedGemm wg;
        wg.M = D; wg.N = D; wg.K = M; wg.groups = 2; wg.TA = true; wg.lda = wg.ldb = wg.ldc = D; wg.beta = 1;
        wg.A[0] = sv->h; wg.B[0] = sc->d_z; wg.C[0] = gw->w2;
        wg.A[1] = x; wg.B[1] = sc->d_h; wg.C[1] = gw->w1;
        TRY(launch_gemm_umma_grouped(wg, br.fork(0)));
    }
    TRY(launch_gemm(M, D, D, sc->d_h, D, false, w->w1, D, true, nullptr, 0, nullptr, 1, 0, d_x, D, s));
    return br.join_deferrable();
}

API int bdetr_decoder_self_fwd(int B, int Q, int D, int H, const float *q0, const float *q0_tc, const bdetr_attn_params *w,
                               float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev, float ln_eps,
                               int training, float *out, const bdetr_attn_saved *sv, float *mha, void *stream)
{
    BDETR_REQUIRE(B > 0 && Q > 0 && D == 256 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(q0 && w && out && sv && mha && sv->qp && sv->kp && sv->vp && sv->o && sv->lse && sv->mean && sv->rstd, BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const float *qin = q0_tc ? q0_tc : q0;
    // [1,Q,D]: projections (one grouped GEMM), attention core, output projection depend on the query parameter only
    const Proj p[3] = {{w->wq, w->bq, sv->qp}, {w->wk, w->bk, sv->kp}, {w->wv, w->bv, sv->vp}};
    const float *tab[3] = {nullptr, nullptr, nullptr};
    TRY(proj_group_fwd(Q, D, qin, 3, p, tab, Q, s));
    TRY(launch_attention_fwd(1, H, Q, Q, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, 1, s));
    {
        GroupedGemm g;
        g.M = Q; g.N = D; g.K = D; g.lda = g.ldb = g.ldc = D;
        g.A[0] = sv->o; g.B[0] = w->wo; g.bias[0] = w->bo; g.C[0] = mha;
        TRY(launch_gemm_umma_grouped(g, s));
    }
    // per image: Dropout (its own mask) + residual + LayerNorm
    TRY(launch_res_ln_bcast_fwd(B * Q, Q, D, q0, mha, training ? sv->z : nullptr, w->ln_gamma, w->ln_beta, ln_eps, dropout_rate, dropout_key,
                                dropout_seed_dev, out, sv->mean, sv->rstd, 1, s));
    return BDETR_OK;
}

API int bdetr_decoder_self_bwd(int B, int Q, int D, int H, const float *q0, const float *q0_tc, const bdetr_attn_params *w,
                               float dropout_rate, uint32_t dropout_key, const uint32_t *dropout_seed_dev,
                               const bdetr_attn_saved *sv, const float *d_out, float *d_q0,
                               const bdetr_attn_params *gw, const bdetr_attn_scratch *sc, float *d_resid, float *sums,
                               void *stream)
{
    BDETR_REQUIRE(B > 0 && Q > 0 && D == 256 && H > 0 && D % H == 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(q0 && w && sv && d_out && sc && d_resid && sums, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(sc->d_qp && sc->d_kp && sc->d_vp && sc->d_o && sc->d_z && sc->delta, BDETR_E_NULL, "null scratch buffer");
    if (!d_q0 && !gw) return BDETR_OK;
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const float *qin = q0_tc ? q0_tc : q0;
    TRY(launch_res_ln_bwd(B * Q, D, d_out, sv->z, sv->mean, sv->rstd, w->ln_gamma, dropout_rate, dropout_key, dropout_seed_dev,
                          d_resid, 0, sc->d_z, gw ? gw->ln_gamma : nullptr, gw ? gw->ln_beta : nullptr, gw ? gw->bo : nullptr, 0, s));
    // sum over the batch: gradient of the shared [Q,D] residual and of the shared attention output
    float *S_r = sums, *S_a = sums + (size_t)Q * D;
    BatchReduce r;
    r.B = B; r.D = D; r.n = 2;
    r.src[0] = d_resid; r.rows[0] = Q; r.sum[0] = S_r;
    r.src[1] = sc->d_z; r.rows[1] = Q; r.sum[1] = S_a;
    TRY(launch_batch_reduce(r, s));
    Branches br(s);
    if (gw) TRY(launch_gemm(D, D, Q, sv->o, D, true, S_a, D, false, nullptr, 0, nullptr, 1, 0, gw->wo, D, br.fork(0)));
    {
        GroupedGemm g;                                   // d_o = d_mha Wo^T
        g.M = Q; g.N = D; g.K = D; g.TB = true; g.lda = g.ldb = g.ldc = D; g.round_out = 1;
        g.A[0] = S_a; g.B[0] = w->wo; g.C[0] = sc->d_o;
        TRY(launch_gemm_umma_grouped(g, s));
    }
    TRY(launch_attention_bwd(1, H, Q, Q, D / H, sv->qp, sv->kp, sv->vp, sv->o, sv->lse, sc->d_o, sc->delta,
                             sc->d_qp, sc->d_kp, sc->d_vp, 1, s));
    const float *dY[3] = {sc->d_qp, sc->d_kp, sc->d_vp};
    const float *Wm[3] = {w->wq, w->wk, w->wv};
    if (gw) {
        float *gW[3] = {gw->wq, gw->wk, gw->wv};
        cudaStream_t ws = br.fork(1);
        TRY(proj_group_wgrad(Q, D, qin, 3, dY, gW, ws));
        BatchReduce cb;                                  // bias gradients: column sums of the [Q,D] projected-tensor gradients
        cb.B = 1; cb.D = D; cb.n = 3;
        cb.src[0] = sc->d_qp; cb.rows[0] = Q; cb.colsum[0] = gw->bq;
        cb.src[1] = sc->d_kp; cb.rows[1] = Q; cb.colsum[1] = gw->bk;
        cb.src[2] = sc->d_vp; cb.rows[2] = Q; cb.colsum[2] = gw->bv;
        TRY(launch_batch_reduce(cb, ws));
    }
    if (d_q0) TRY(proj_group_dgrad(Q, D, 3, dY, Wm, S_r, Q, d_q0, 1, s));     // d_q0 += S_r + sum_g dY[g] W[g]^T
    return br.join_deferrable();
}

// ---- workspace queries (caller-owned buffers; see include/bdetr.h) ------------------------------------------------------
API size_t bdetr_attention_block_saved_bytes(int B, int Lq, int Lk, int D, int H, int training)
{
    const size_t q = (size_t)B * Lq * D, k = (size_t)B * Lk * D;
    return 4 * (q + 2 * k + q /* o */ + (size_t)B * H * Lq /* lse */ + (training ? q : 0) /* z */ + 2 * (size_t)B * Lq /* mean, rstd */);
}
API size_t bdetr_attention_block_scratch_bytes(int B, int Lq, int Lk, int D, int H)
{
    const size_t q = (size_t)B * Lq * D, k = (size_t)B * Lk * D;
    const size_t L = (size_t)(Lq > Lk ? Lq : Lk);
    return 4 * (q + 2 * k /* d_qp, d_kp, d_vp */ + q /* d_o */ + q /* d_z */ + (size_t)B * H * Lq /* delta */ + q /* d_resid */ + 4 * L * D /* sums */);
}
API size_t bdetr_ffn_block_saved_bytes(int M, int D, int training) { return 4 * ((size_t)M * D * (training ? 2 : 1) + 2 * (size_t)M); }
API size_t bdetr_ffn_block_scratch_bytes(int M, int D) { return 4 * 2 * (size_t)M * D; }
API size_t bdetr_heads_saved_bytes(int M, int Dh, int C, int A)
{
    return 4 * (3 * (size_t)M * Dh + 4 * 3 * (size_t)Dh + (size_t)((M + 127) / 128) * 2 * 3 * Dh + (size_t)M * (C + A + 4));
}
API size_t bdetr_heads_scratch_bytes(int M, int Dh, int C, int A)
{
    const size_t n = (size_t)C + A + 4;
    return 4 * ((size_t)M * n + (size_t)Dh * n + n + 2 * 3 * (size_t)Dh + 3 * (size_t)M * Dh);
}
