// The three prediction heads of one boosted block in one call (include/bdetr.h bdetr_heads_fwd / bdetr_heads_bwd).
// Reference: prediction_heads.py:46-63 (box), :113-131 (category), :182-201 (attribute); boosted_model.py:222-229 (running sum).
//   hidden layers      ONE grouped tcgen05 GEMM  h[k] = relu(x W1[k] + b1[k])                       (k = category, attribute, box)
//   BatchNorm          statistics by a deterministic two-level column reduction; the normalisation itself is folded into
//                      the second Dense:  ((h - mu) rstd gamma + beta) W2 + b2 = h (diag(rstd gamma) W2) + ((beta - mu rstd gamma) W2 + b2)
//   second Dense + activation + boosted running sum: one fp32 kernel, every row evaluated by the same instruction sequence
//                      (identical query rows give bit-identical predictions: the matcher's tie rule depends on it)
// Backward: G = h^T d_logits and colsum(d_logits) give the second-layer gradients AND both BatchNorm reduction terms
// (sum d_hn = W2 colsum(d), sum d_hn xhat = rowsum(W2 * xhat^T d)), so hn / d_hn are never materialised.
#include <math_constants.h>
#include "umma.cuh"

using namespace bdetr;
#define API extern "C" __attribute__((visibility("default")))
#define TRY(x) do { int rc__ = (x); if (rc__ != BDETR_OK) return rc__; } while (0)

namespace bdetr {

struct HeadsDims { int M, Dh, n[3], off[3], ntot; };       // off[k] = first column of head k in the concatenated [.., C+A+4] layouts

struct HeadsFoldArgs {
    HeadsDims d;
    const float *h;                                          // [3,M,Dh]
    const float *gamma[3], *beta[3], *w2[3], *b2[3];
    float *moving_mean[3], *moving_var[3];
    int training[3];
    float eps, momentum;
    const float *part;                                       // [chunks][2][3*Dh] partial sums (pivoted)
    int chunks;
    float *bn_mean, *bn_rstd;                                // [3,Dh]
    float *w2f, *b2f;                                        // [Dh * ntot] (head k at Dh*off[k], row stride n[k]), [ntot]
};

// partial column sums of h over 128-row chunks, pivoted on row 0 (kills the cancellation in E[x^2] - mean^2)
__global__ void __launch_bounds__(256)
heads_bn_stats_kernel(int M, int cols, const float *__restrict__ h0, size_t head_stride, int Dh, float *__restrict__ part)
{
    pdl_sync();
    __shared__ float red[8][33];
    const int gc = blockIdx.x * 32 + (threadIdx.x & 31), r = threadIdx.x >> 5;      // gc = column in [0, 3*Dh)
    const bool live = gc < cols;
    const int k = live ? gc / Dh : 0, c = live ? gc % Dh : 0;
    const float *h = h0 + (size_t)k * head_stride;
    const int m0 = blockIdx.y * 128, m1 = min(M, m0 + 128);
    const float pivot = live ? h[c] : 0.0f;
    float s1 = 0.0f, s2 = 0.0f;
    if (live) for (int m = m0 + r; m < m1; m += 8) { const float d = h[(size_t)m * Dh + c] - pivot; s1 += d; s2 = fmaf(d, d, s2); }
    __syncthreads(); red[r][threadIdx.x & 31] = s1; __syncthreads();
    float t1 = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t1 += red[j][threadIdx.x & 31];
    __syncthreads(); red[r][threadIdx.x & 31] = s2; __syncthreads();
    float t2 = 0.0f;
#pragma unroll
    for (int j = 0; j < 8; ++j) t2 += red[j][threadIdx.x & 31];
    if (live && r == 0) { part[((size_t)blockIdx.y * 2) * cols + gc] = t1; part[((size_t)blockIdx.y * 2 + 1) * cols + gc] = t2; }
}

// grid (3 heads), thread = hidden column: statistics -> mean / rstd, moving-statistics update, and the affine map
// hn = h * scale + shift (scale = rstd gamma, shift = beta - mean scale) the output kernel folds into the second Dense
__global__ void __launch_bounds__(256)
heads_bn_finalize_kernel(HeadsFoldArgs a)
{
    pdl_sync();
    const int k = blockIdx.x, Dh = a.d.Dh, c = threadIdx.x;
    if (c >= Dh) return;
    float mean, var;
    if (a.training[k]) {
        float t1 = 0.0f, t2 = 0.0f;
        const int cols = 3 * Dh, gc = k * Dh + c;
        for (int j = 0; j < a.chunks; ++j) { t1 += a.part[((size_t)j * 2) * cols + gc]; t2 += a.part[((size_t)j * 2 + 1) * cols + gc]; }   // fixed order
        const float a1 = t1 / (float)a.d.M, a2 = t2 / (float)a.d.M;
        mean = a.h[(size_t)k * a.d.M * Dh + c] + a1;
        var = fmaxf(a2 - a1 * a1, 0.0f);
        a.moving_mean[k][c] = a.moving_mean[k][c] * a.momentum + mean * (1.0f - a.momentum);
        a.moving_var[k][c] = a.moving_var[k][c] * a.momentum + var * (1.0f - a.momentum);
    } else {
        mean = a.moving_mean[k][c];
        var = a.moving_var[k][c];
    }
    const float rstd = rsqrtf(var + a.eps);
    a.bn_mean[k * Dh + c] = mean;
    a.bn_rstd[k * Dh + c] = rstd;
    const float sc = rstd * a.gamma[k][c];
    a.w2f[k * Dh + c] = sc;                               // scale [3,Dh]
    a.b2f[k * Dh + c] = a.beta[k][c] - mean * sc;         // shift [3,Dh]
}

struct HeadsOutArgs {
    HeadsDims d;
    const float *h, *scale, *shift;                       // [3,M,Dh], [3,Dh], [3,Dh]
    const float *w2[3], *b2[3];
    float mult;
    const float *cum_in[3]; float *cum_out[3]; float *act[3];
};
constexpr int HO_ROWS = 32, HO_RPW = 4, HO_WBUF = 44 * 1024, HO_THREADS = 256;   // rows per CTA, rows per warp, bytes per W2 chunk buffer
// Heads wider than HO_SLAB outputs: column slabs of HO_SLAB, W2 rows staged at stride HO_SLDW (the slab plus the
// 16-byte alignment slack on both sides), HO_SCK rows per chunk (one bulk copy per lane of warp 0)
constexpr int HO_SLAB = 320, HO_SLDW = HO_SLAB + 8, HO_SCK = 32, HO_MAXN = 2048;
static_assert(HO_SCK * HO_SLDW * 4 <= HO_WBUF, "slab chunk must fit one W2 buffer");

__device__ __forceinline__ float sigmoidf_h(float x) { return 1.0f / (1.0f + expf(-x)); }

// 1-D bulk copy global -> shared through the TMA engine, completion on an mbarrier (16-byte aligned, size % 16 == 0)
__device__ __forceinline__ void bulk_load_1d(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}

// Slab path: W2 rows c1 .. c1 + ck - 1 (ck <= 32), columns [n0, n0 + w), into dst at row stride HO_SLDW.  A slab row is
// not 16-byte aligned in general (row stride N), so lane i copies the aligned span that covers row c1 + i; the slab
// starts (c N + n0) & 3 floats into it.  The span never passes the end of W2: Dh N is a multiple of 4.
__device__ __forceinline__ void heads_slab_chunk(const float *w2, int N, int n0, int w, int c1, int ck, float *dst, uint64_t *bar)
{
    const int lane = threadIdx.x & 31;
    size_t s0 = 0;
    uint32_t bytes = 0;
    if (lane < ck) {
        const size_t st = (size_t)(c1 + lane) * N + n0;
        s0 = st & ~size_t(3);
        bytes = (uint32_t)((((st + w + 3) & ~size_t(3)) - s0) * 4);
    }
    const uint32_t total = __reduce_add_sync(0xffffffffu, bytes);
    if (lane == 0) mbar_expect_tx(bar, total);
    __syncwarp();
    if (lane < ck) bulk_load_1d(dst + lane * HO_SLDW, w2 + s0, bytes, bar);
}

// rows of this warp (HO_RPW + the shift row) x NJ output columns per lane, W2 streamed in row chunks of CK hidden units.
// SLAB: columns [n0, n0 + w) of a wider head (CK = HO_SCK); the raw logits go to act, the row activation runs after.
template <int NJ, bool SLAB = false>
__device__ __forceinline__ void heads_out_rows(const HeadsOutArgs &a, int k, int N, int M, int Dh, int m0, const float *sH, float *sWbuf,
                                               uint64_t *bars, int CK, int n0 = 0, int w = 0)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const float *w2 = a.w2[k];
    float acc[HO_RPW + 1][NJ];
#pragma unroll
    for (int r = 0; r <= HO_RPW; ++r)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[r][j] = 0.0f;
    const float *hr = sH + (warp * HO_RPW) * Dh, *hs = sH + HO_ROWS * Dh;
    const int nchunks = (Dh + CK - 1) / CK;
    const int ldw = SLAB ? HO_SLDW : N;
    int off[4] = {0, 0, 0, 0};                                // SLAB: where the slab starts in a staged row (chunks start at multiples of 4 rows)
    if (SLAB) {
#pragma unroll
        for (int cc = 0; cc < 4; ++cc) off[cc] = (cc * N + n0) & 3;
        if (warp == 0) heads_slab_chunk(w2, N, n0, w, 0, min(CK, Dh), sWbuf, &bars[0]);
    } else if (threadIdx.x == 0) {
        const int ck = min(CK, Dh);
        mbar_expect_tx(&bars[0], (uint32_t)(ck * N * 4));
        bulk_load_1d(sWbuf, w2, (uint32_t)(ck * N * 4), &bars[0]);
    }
    for (int ch = 0; ch < nchunks; ++ch) {
        const int c0 = ch * CK, ck = min(CK, Dh - c0);
        if (SLAB) {
            if (warp == 0 && ch + 1 < nchunks)
                heads_slab_chunk(w2, N, n0, w, c0 + CK, min(CK, Dh - c0 - CK),
                                 reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(sWbuf) + ((ch + 1) & 1) * HO_WBUF), &bars[(ch + 1) & 1]);
        } else if (threadIdx.x == 0 && ch + 1 < nchunks) {   // next chunk into the other buffer (its readers passed the barrier below)
            const int c1 = c0 + CK, ck1 = min(CK, Dh - c1);
            mbar_expect_tx(&bars[(ch + 1) & 1], (uint32_t)(ck1 * N * 4));
            bulk_load_1d(reinterpret_cast<uint8_t *>(sWbuf) + ((ch + 1) & 1) * HO_WBUF, w2 + (size_t)c1 * N, (uint32_t)(ck1 * N * 4), &bars[(ch + 1) & 1]);
        }
        mbar_wait(&bars[ch & 1], (ch >> 1) & 1);
        const float *sW = reinterpret_cast<const float *>(reinterpret_cast<const uint8_t *>(sWbuf) + (ch & 1) * HO_WBUF);
        for (int c = 0; c < ck; c += 4) {                     // the SAME summation order for every row: identical rows stay bit-identical
            float4 hv[HO_RPW + 1];
#pragma unroll
            for (int r = 0; r < HO_RPW; ++r) hv[r] = *reinterpret_cast<const float4 *>(hr + r * Dh + c0 + c);
            hv[HO_RPW] = *reinterpret_cast<const float4 *>(hs + c0 + c);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc) {
                const float *wrow = sW + (c + cc) * ldw + off[cc] + lane;
                float w[NJ];
#pragma unroll
                for (int j = 0; j < NJ; ++j) w[j] = wrow[32 * j];           // (columns >= N read the next row / slack: discarded below)
#pragma unroll
                for (int r = 0; r <= HO_RPW; ++r) {
                    const float hvv = cc == 0 ? hv[r].x : cc == 1 ? hv[r].y : cc == 2 ? hv[r].z : hv[r].w;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) acc[r][j] = fmaf(hvv, w[j], acc[r][j]);
                }
            }
        }
        __syncthreads();                                      // everyone is done with buffer ch & 1 before it is refilled
    }
    // logits = acc[row] + (shift W2 + b2); activation; running sum
    float bb[NJ];
    if (SLAB) {
#pragma unroll
        for (int j = 0; j < NJ; ++j) bb[j] = (lane + 32 * j < w) ? a.b2[k][n0 + lane + 32 * j] + acc[HO_RPW][j] : 0.0f;
#pragma unroll
        for (int r = 0; r < HO_RPW; ++r) {
            const int m = m0 + warp * HO_RPW + r;
            if (m >= M) continue;
#pragma unroll
            for (int j = 0; j < NJ; ++j)
                if (lane + 32 * j < w) a.act[k][(size_t)m * N + n0 + lane + 32 * j] = acc[r][j] + bb[j];
        }
        return;
    }
#pragma unroll
    for (int j = 0; j < NJ; ++j) bb[j] = (lane + 32 * j < N) ? a.b2[k][lane + 32 * j] + acc[HO_RPW][j] : 0.0f;
#pragma unroll
    for (int r = 0; r < HO_RPW; ++r) {
        const int m = m0 + warp * HO_RPW + r;
        if (m >= M) continue;
        float p[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) p[j] = acc[r][j] + bb[j];
        if (k == 0) {                                      // softmax over the whole row
            float mx = -CUDART_INF_F;
#pragma unroll
            for (int j = 0; j < NJ; ++j) if (lane + 32 * j < N) mx = fmaxf(mx, p[j]);
            mx = warp_max(mx);
            float sm = 0.0f;
#pragma unroll
            for (int j = 0; j < NJ; ++j) { p[j] = (lane + 32 * j < N) ? expf(p[j] - mx) : 0.0f; sm += p[j]; }
            sm = warp_sum(sm);
#pragma unroll
            for (int j = 0; j < NJ; ++j) p[j] = p[j] / sm;
        } else {
#pragma unroll
            for (int j = 0; j < NJ; ++j) p[j] = k == 1 ? sigmoidf_h(p[j]) : 3.0f * sigmoidf_h(p[j] / 100.0f) - 1.0f;
        }
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int n = lane + 32 * j;
            if (n < N) {
                const size_t o = (size_t)m * N + n;
                a.act[k][o] = p[j];
                a.cum_out[k][o] = (a.cum_in[k] ? a.cum_in[k][o] : 0.0f) + a.mult * p[j];
            }
        }
    }
}

// Second Dense + activation + boosted running sum.  grid (row tiles of 32, 3 heads), 8 warps; warp = 4 rows, lane = output
// columns lane, lane + 32, ...  BatchNorm is applied while the rows are staged (sH = h * scale; one extra row holds
// `shift`, whose product with W2 is the folded bias), so hn is never materialised.  W2 [Dh, N] arrives in row chunks by TMA
// bulk copies (double-buffered).  dynamic smem: bars | sH [33][Dh] | sW 2 x 44 KB (+ slack)
// SLABS (some head has more than HO_SLAB outputs): grid.z = column slabs.  A head that wide gets its raw logits, slab by
// slab, from every z; a narrower head runs the whole-row path above in z = 0 only.
template <bool SLABS>
__global__ void __launch_bounds__(HO_THREADS)
heads_out_kernel(HeadsOutArgs a)
{
    extern __shared__ __align__(128) uint8_t smem_b[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_b);
    const int k = blockIdx.y, Dh = a.d.Dh, N = a.d.n[k], M = a.d.M;
    const int n0 = SLABS ? blockIdx.z * HO_SLAB : 0;
    if (SLABS && (N > HO_SLAB ? n0 >= N : blockIdx.z != 0)) return;
    float *sH = reinterpret_cast<float *>(smem_b + 128);
    float *sW = sH + (HO_ROWS + 1) * Dh;
    if (threadIdx.x == 0) {
        mbar_init(&bars[0], 1); mbar_init(&bars[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    pdl_sync();
    const int m0 = blockIdx.x * HO_ROWS;
    const float *h = a.h + (size_t)k * M * Dh;
    const float *scale = a.scale + k * Dh, *shift = a.shift + k * Dh;
    for (int e = threadIdx.x; e < (HO_ROWS + 1) * Dh / 4; e += HO_THREADS) {
        const int r = e / (Dh / 4), c4 = e % (Dh / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r == HO_ROWS) v = *reinterpret_cast<const float4 *>(shift + 4 * c4);
        else if (m0 + r < M) {
            v = *reinterpret_cast<const float4 *>(h + (size_t)(m0 + r) * Dh + 4 * c4);
            const float4 sc = *reinterpret_cast<const float4 *>(scale + 4 * c4);
            v.x *= sc.x; v.y *= sc.y; v.z *= sc.z; v.w *= sc.w;
        }
        *reinterpret_cast<float4 *>(sH + r * Dh + 4 * c4) = v;
    }
    __syncthreads();
    if (SLABS && N > HO_SLAB) {
        heads_out_rows<10, true>(a, k, N, M, Dh, m0, sH, sW, bars, HO_SCK, n0, min(HO_SLAB, N - n0));
        return;
    }
    // rows of W2 per chunk: a multiple of 4 (16-byte sized / aligned copies) that fits one 48 KB buffer
    const int CK = max(4, min(Dh, (HO_WBUF / (N * 4)) & ~3));
    if (N <= 32) heads_out_rows<1>(a, k, N, M, Dh, m0, sH, sW, bars, CK);
    else if (N <= 96) heads_out_rows<3>(a, k, N, M, Dh, m0, sH, sW, bars, CK);
    else heads_out_rows<10>(a, k, N, M, Dh, m0, sH, sW, bars, CK);
}

// ---- backward ---------------------------------------------------------------------------------------------------------
struct HeadsActBwdArgs {
    HeadsDims d; float mult;
    const float *act[3]; const float *d_cum[3];
    float *d_logits;                 // head k at M*off[k], row stride n[k]
    float *colsum_d;                 // [ntot] += column sums of d_logits (pre-zeroed)
};
// grid (row tiles of 32, 3 heads); one warp per row, 4 rows per warp; column sums through shared memory
__global__ void __launch_bounds__(256)
heads_act_bwd_kernel(HeadsActBwdArgs a)
{
    pdl_sync();
    extern __shared__ float s_cs[];                   // [max N]
    const int k = blockIdx.y, N = a.d.n[k], M = a.d.M;
    for (int n = threadIdx.x; n < N; n += 256) s_cs[n] = 0.0f;
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float *dl = a.d_logits + (size_t)M * a.d.off[k];
    for (int r = warp; r < 32; r += 8) {
        const int m = blockIdx.x * 32 + r;
        if (m >= M) break;
        const float *p = a.act[k] + (size_t)m * N, *g = a.d_cum[k] + (size_t)m * N;
        float *d = dl + (size_t)m * N;
        if (k == 0) {
            float dot = 0.0f;
            for (int n = lane; n < N; n += 32) dot = fmaf(g[n], p[n], dot);
            dot = warp_sum(dot);
            for (int n = lane; n < N; n += 32) { const float v = a.mult * p[n] * (g[n] - dot); d[n] = v; atomicAdd(&s_cs[n], v); }
        } else if (k == 1) {
            for (int n = lane; n < N; n += 32) { const float v = a.mult * g[n] * p[n] * (1.0f - p[n]); d[n] = v; atomicAdd(&s_cs[n], v); }
        } else {
            for (int n = lane; n < N; n += 32) {
                const float sg = (p[n] + 1.0f) / 3.0f;
                const float v = a.mult * g[n] * 3.0f * sg * (1.0f - sg) / 100.0f;
                d[n] = v; atomicAdd(&s_cs[n], v);
            }
        }
    }
    __syncthreads();
    for (int n = threadIdx.x; n < N; n += 256) atomicAdd(&a.colsum_d[a.d.off[k] + n], s_cs[n]);
}

struct HeadsBnBwdArgs {
    HeadsDims d;
    const float *hTd;                // head k at Dh*off[k]: [Dh, n[k]] = h^T d_logits
    const float *colsum_d;           // [ntot]
    const float *bn_mean, *bn_rstd;  // [3,Dh]
    const float *gamma[3], *beta[3], *w2[3];
    int training[3];
    float *g_w2[3], *g_b2[3], *g_gamma[3], *g_beta[3];      // all NULL for a frozen head
    float *bn_s;                     // [2][3][Dh]: s1 = sum_m d_hn, s2 = sum_m d_hn xhat (zero when the BN ran on moving statistics)
};
// grid (Dh / 8, 3 heads), one WARP per hidden column, lane = output column: coalesced rows of G and W2, warp sums
__global__ void __launch_bounds__(256)
heads_bn_bwd_kernel(HeadsBnBwdArgs a)
{
    pdl_sync();
    const int k = blockIdx.y, Dh = a.d.Dh, N = a.d.n[k];
    const int lane = threadIdx.x & 31, c = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (c < Dh) {
        const float mu = a.bn_mean[k * Dh + c], rstd = a.bn_rstd[k * Dh + c], gam = a.gamma[k][c], bet = a.beta[k][c];
        const float *G = a.hTd + (size_t)Dh * a.d.off[k] + (size_t)c * N;
        const float *w2 = a.w2[k] + (size_t)c * N;
        const float *cs = a.colsum_d + a.d.off[k];
        float *gw2 = a.g_w2[k] ? a.g_w2[k] + (size_t)c * N : nullptr;
        float s1 = 0.0f, s2 = 0.0f;
        for (int n = lane; n < N; n += 32) {
            const float csn = cs[n], w = w2[n];
            const float xd = rstd * (G[n] - mu * csn);            // (xhat^T d)[c,n]
            s1 = fmaf(csn, w, s1);
            s2 = fmaf(w, xd, s2);
            if (gw2) gw2[n] += gam * xd + bet * csn;              // hn^T d
        }
        s1 = warp_sum(s1); s2 = warp_sum(s2);
        if (lane == 0) {
            if (a.g_gamma[k]) { a.g_gamma[k][c] += s2; a.g_beta[k][c] += s1; }
            a.bn_s[(0 * 3 + k) * Dh + c] = a.training[k] ? s1 : 0.0f;
            a.bn_s[(1 * 3 + k) * Dh + c] = a.training[k] ? s2 : 0.0f;
        }
    }
    if (blockIdx.x == 0 && a.g_b2[k]) for (int n = threadIdx.x; n < N; n += 256) a.g_b2[k][n] += a.colsum_d[a.d.off[k] + n];
}

struct HeadsDhArgs {
    HeadsDims d;
    const float *h, *d_logits;       // [3,M,Dh]; concatenated d_logits
    const float *w2[3], *gamma[3];
    const float *bn_mean, *bn_rstd, *bn_s;
    float *d_h;                      // [3,M,Dh], stored tf32-rounded (feeds the tcgen05 dgrad / wgrad GEMMs)
    float *g_b1[3];                  // += column sums of d_h (NULL: frozen)
};
// d_h = relu'(h) gamma rstd (d_logits W2^T - s1/M - xhat s2/M).  grid (row tiles of 16, 3 heads), thread = hidden column c:
// it walks ITS row of W2 against the tile's d_logits rows staged in shared memory (broadcast LDS.128 along n), 16
// accumulators.  W2 [Dh, N] is pulled into shared memory whole by one TMA bulk copy when it fits (DH_WMAX bytes), else
// each thread reads its (contiguous) row through L1.  dynamic smem: bar | sD [16][Np] | sW [Dh*N]
constexpr int DH_ROWS = 16, DH_WMAX = 96 * 1024;
__global__ void __launch_bounds__(256)
heads_dh_kernel(HeadsDhArgs a)
{
    extern __shared__ __align__(128) uint8_t smem_b[];
    uint64_t *bar = reinterpret_cast<uint64_t *>(smem_b);
    const int k = blockIdx.y, Dh = a.d.Dh, N = a.d.n[k], M = a.d.M, c = threadIdx.x;
    const int Np = (N + 3) & ~3;
    const int npmax = (max(max(a.d.n[0], a.d.n[1]), a.d.n[2]) + 3) & ~3;
    float *sD = reinterpret_cast<float *>(smem_b + 128);
    float *sW = sD + DH_ROWS * npmax;
    const bool w_in_smem = Dh * N * 4 <= DH_WMAX;
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    pdl_sync();
    if (threadIdx.x == 0 && w_in_smem) {
        mbar_expect_tx(bar, (uint32_t)(Dh * N * 4));
        bulk_load_1d(sW, a.w2[k], (uint32_t)(Dh * N * 4), bar);
    }
    const int m0 = blockIdx.x * DH_ROWS;
    const float *dl = a.d_logits + (size_t)M * a.d.off[k];
    for (int e = threadIdx.x; e < DH_ROWS * Np; e += 256) {
        const int r = e / Np, n = e % Np;
        sD[e] = (m0 + r < M && n < N) ? dl[(size_t)(m0 + r) * N + n] : 0.0f;
    }
    __syncthreads();
    if (w_in_smem) mbar_wait(bar, 0);
    float acc[DH_ROWS];
#pragma unroll
    for (int r = 0; r < DH_ROWS; ++r) acc[r] = 0.0f;
    if (c < Dh) {
        const float *wrow = (w_in_smem ? sW : a.w2[k]) + (size_t)c * N;
        for (int n = 0; n < Np; n += 4) {
            const float w0 = wrow[n], w1 = n + 1 < N ? wrow[n + 1] : 0.0f, w2v = n + 2 < N ? wrow[n + 2] : 0.0f, w3 = n + 3 < N ? wrow[n + 3] : 0.0f;
#pragma unroll
            for (int r = 0; r < DH_ROWS; ++r) {
                const float4 d4 = *reinterpret_cast<const float4 *>(sD + r * Np + n);
                acc[r] = fmaf(d4.x, w0, fmaf(d4.y, w1, fmaf(d4.z, w2v, fmaf(d4.w, w3, acc[r]))));
            }
        }
    }
    if (c >= Dh) return;
    const float mu = a.bn_mean[k * Dh + c], rstd = a.bn_rstd[k * Dh + c], g = a.gamma[k][c];
    const float invM = 1.0f / (float)M;
    const float s1 = a.bn_s[(0 * 3 + k) * Dh + c] * invM, s2 = a.bn_s[(1 * 3 + k) * Dh + c] * invM;
    const float *h = a.h + (size_t)k * M * Dh;
    float *dh = a.d_h + (size_t)k * M * Dh;
    float bsum = 0.0f;
#pragma unroll
    for (int r = 0; r < DH_ROWS; ++r) {
        const int m = m0 + r;
        if (m < M) {
            const float hv = h[(size_t)m * Dh + c];
            const float xh = (hv - mu) * rstd;
            const float o = hv > 0.0f ? tf32_rn(g * rstd * (acc[r] - s1 - xh * s2)) : 0.0f;
            dh[(size_t)m * Dh + c] = o;
            bsum += o;
        }
    }
    if (a.g_b1[k]) atomicAdd(&a.g_b1[k][c], bsum);
}

static bool heads_dims(HeadsDims &d, int M, int Dh, int C, int A)
{
    d.M = M; d.Dh = Dh; d.n[0] = C; d.n[1] = A; d.n[2] = 4;
    d.off[0] = 0; d.off[1] = C; d.off[2] = C + A; d.ntot = C + A + 4;
    return M > 0 && Dh > 0 && Dh <= 256 && Dh % 4 == 0 && C > 0 && A > 0;
}

}  // namespace bdetr

API int bdetr_heads_fwd(int M, int D, int Dh, int C, int A, const float *x, const bdetr_head_params *heads,
                        const int *bn_training, float bn_eps, float bn_momentum, float mult,
                        const float *const *cum_in, float *const *cum_out, const bdetr_heads_saved *sv, void *stream)
{
    HeadsDims d;
    BDETR_REQUIRE(heads_dims(d, M, Dh, C, A) && D > 0 && D % 4 == 0, BDETR_E_BAD_SHAPE, "bad shape (hidden width <= 256)");
    BDETR_REQUIRE(C <= HO_MAXN && A <= HO_MAXN, BDETR_E_UNSUPPORTED, "fused heads: at most 2048 outputs per head");
    BDETR_REQUIRE(x && heads && bn_training && cum_out && sv && sv->h && sv->bn_mean && sv->bn_rstd && sv->bn_part && sv->w2f && sv->b2f, BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const size_t hs = (size_t)M * Dh;
    GroupedGemm g;
    g.M = M; g.N = Dh; g.K = D; g.groups = 3; g.share_a = true; g.lda = D; g.ldb = Dh; g.ldc = Dh; g.act = 1;
    g.A[0] = x;
    for (int k = 0; k < 3; ++k) { g.B[k] = heads[k].w1; g.bias[k] = heads[k].b1; g.C[k] = sv->h + k * hs; }
    TRY(launch_gemm_umma_grouped(g, s));
    const int chunks = ceil_div(M, 128);
    float *part = sv->bn_part;
    const bool any_training = bn_training[0] || bn_training[1] || bn_training[2];
    if (any_training) {
        launch_k(heads_bn_stats_kernel, dim3(ceil_div(3 * Dh, 32), chunks), 256, 0, s, M, 3 * Dh, (const float *)sv->h, hs, Dh, part);
        BDETR_CHECK_LAUNCH("heads_bn_stats_kernel");
    }
    HeadsFoldArgs f;
    f.d = d; f.h = sv->h; f.eps = bn_eps; f.momentum = bn_momentum; f.part = part; f.chunks = chunks;
    f.bn_mean = sv->bn_mean; f.bn_rstd = sv->bn_rstd; f.w2f = sv->w2f; f.b2f = sv->b2f;
    for (int k = 0; k < 3; ++k) {
        f.gamma[k] = heads[k].bn_gamma; f.beta[k] = heads[k].bn_beta; f.w2[k] = heads[k].w2; f.b2[k] = heads[k].b2;
        f.moving_mean[k] = heads[k].bn_moving_mean; f.moving_var[k] = heads[k].bn_moving_var; f.training[k] = bn_training[k];
    }
    launch_k(heads_bn_finalize_kernel, dim3(3), 256, 0, s, f);
    BDETR_CHECK_LAUNCH("heads_bn_finalize_kernel");
    HeadsOutArgs o;
    o.d = d; o.h = sv->h; o.scale = sv->w2f; o.shift = sv->b2f; o.mult = mult;
    for (int k = 0; k < 3; ++k) {
        o.w2[k] = heads[k].w2; o.b2[k] = heads[k].b2;
        o.cum_in[k] = cum_in ? cum_in[k] : nullptr; o.cum_out[k] = cum_out[k]; o.act[k] = sv->act[k];
    }
    const size_t smem = 128 + (size_t)(HO_ROWS + 1) * Dh * sizeof(float) + 2 * HO_WBUF + 2048;
    const int slabs = ceil_div(max(C, A), HO_SLAB);
    auto kern = slabs > 1 ? heads_out_kernel<true> : heads_out_kernel<false>;
    static size_t optin[2] = {0, 0};
    if (smem > optin[slabs > 1]) {
        BDETR_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        optin[slabs > 1] = smem;
    }
    launch_k(kern, dim3(ceil_div(M, HO_ROWS), 3, slabs), HO_THREADS, smem, s, o);
    BDETR_CHECK_LAUNCH("heads_out_kernel");
    // heads wider than a slab: activation over the whole row and the running sum, in the per-row order of the layer path
    for (int k = 0; k < 2; ++k) {
        const int n = d.n[k];
        if (n <= HO_SLAB) continue;
        const bool have_in = cum_in && cum_in[k];
        if (have_in && cum_in[k] != cum_out[k])
            BDETR_CUDA(cudaMemcpyAsync(cum_out[k], cum_in[k], sizeof(float) * M * n, cudaMemcpyDeviceToDevice, s));
        TRY(launch_head_act_fwd(M, n, k, mult, sv->act[k], cum_out[k], have_in ? 0 : 1, s));
    }
    return BDETR_OK;
}

API int bdetr_heads_bwd(int M, int D, int Dh, int C, int A, const float *x, const bdetr_head_params *heads,
                        const int *bn_training, float mult, const bdetr_heads_saved *sv, const float *const *d_cum,
                        float *d_x, int accumulate_dx, const bdetr_head_params *const *gw,
                        const bdetr_heads_scratch *sc, void *stream)
{
    HeadsDims d;
    BDETR_REQUIRE(heads_dims(d, M, Dh, C, A) && D > 0 && D % 4 == 0, BDETR_E_BAD_SHAPE, "bad shape (hidden width <= 256)");
    BDETR_REQUIRE(x && heads && bn_training && sv && d_cum && gw && sc && sc->d_logits && sc->hTd && sc->colsum_d && sc->bn_s && sc->d_h,
                  BDETR_E_NULL, "null pointer");
    ModeScope tc(BDETR_MODE_TF32);
    cudaStream_t s = as_stream(stream);
    const size_t hs = (size_t)M * Dh;
    BDETR_CUDA(cudaMemsetAsync(sc->colsum_d, 0, sizeof(float) * d.ntot, s));
    HeadsActBwdArgs ab;
    ab.d = d; ab.mult = mult; ab.d_logits = sc->d_logits; ab.colsum_d = sc->colsum_d;
    for (int k = 0; k < 3; ++k) { ab.act[k] = sv->act[k]; ab.d_cum[k] = d_cum[k]; }
    const int nmax = max(max(C, A), 4);
    launch_k(heads_act_bwd_kernel, dim3(ceil_div(M, 32), 3), 256, sizeof(float) * nmax, s, ab);
    BDETR_CHECK_LAUNCH("heads_act_bwd_kernel");
    // G[k] = h[k]^T d_logits[k]  ([Dh, n_k], contraction over the M rows).  A head wider than a slab takes the fp32
    // GEMM: with tf32 operands the second-layer weight and BatchNorm gamma gradients of a 2048-output head were off by
    // 1e-3 of their largest value (1e-6 in fp32).
    {
        Branches br(s);
        for (int k = 0; k < 3; ++k) {
            ModeScope gm(d.n[k] > HO_SLAB ? BDETR_MODE_FP32 : BDETR_MODE_TF32);
            TRY(launch_gemm(Dh, d.n[k], M, sv->h + k * hs, Dh, true, sc->d_logits + (size_t)M * d.off[k], d.n[k], false, nullptr, 0, nullptr,
                            0, 0, sc->hTd + (size_t)Dh * d.off[k], d.n[k], k == 0 ? s : br.fork(k - 1)));
        }
        TRY(br.join());
    }
    HeadsBnBwdArgs bb;
    bb.d = d; bb.hTd = sc->hTd; bb.colsum_d = sc->colsum_d; bb.bn_mean = sv->bn_mean; bb.bn_rstd = sv->bn_rstd; bb.bn_s = sc->bn_s;
    HeadsDhArgs dh;
    dh.d = d; dh.h = sv->h; dh.d_logits = sc->d_logits; dh.bn_mean = sv->bn_mean; dh.bn_rstd = sv->bn_rstd; dh.bn_s = sc->bn_s; dh.d_h = sc->d_h;
    for (int k = 0; k < 3; ++k) {
        bb.gamma[k] = heads[k].bn_gamma; bb.beta[k] = heads[k].bn_beta; bb.w2[k] = heads[k].w2; bb.training[k] = bn_training[k];
        bb.g_w2[k] = gw[k] ? gw[k]->w2 : nullptr; bb.g_b2[k] = gw[k] ? gw[k]->b2 : nullptr;
        bb.g_gamma[k] = gw[k] ? gw[k]->bn_gamma : nullptr; bb.g_beta[k] = gw[k] ? gw[k]->bn_beta : nullptr;
        dh.w2[k] = heads[k].w2; dh.gamma[k] = heads[k].bn_gamma; dh.g_b1[k] = gw[k] ? gw[k]->b1 : nullptr;
    }
    launch_k(heads_bn_bwd_kernel, dim3(ceil_div(Dh, 8), 3), 256, 0, s, bb);
    BDETR_CHECK_LAUNCH("heads_bn_bwd_kernel");
    const size_t smem = 128 + (size_t)DH_ROWS * ((max(max(C, A), 4) + 3) & ~3) * sizeof(float) + (size_t)min(DH_WMAX, Dh * max(max(C, A), 4) * 4) + 64;
    static size_t optin = 0;
    if (smem > optin) {
        BDETR_CUDA(cudaFuncSetAttribute(heads_dh_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        optin = smem;
    }
    launch_k(heads_dh_kernel, dim3(ceil_div(M, DH_ROWS), 3), 256, smem, s, dh);
    BDETR_CHECK_LAUNCH("heads_dh_kernel");
    Branches br(s);
    {   // gW1[k] += x^T d_h[k]: one grouped weight-gradient GEMM over the heads that train
        GroupedGemm g;
        g.M = D; g.N = Dh; g.K = M; g.share_a = true; g.TA = true; g.lda = D; g.ldb = Dh; g.ldc = Dh; g.beta = 1;
        g.A[0] = x;
        int n = 0;
        for (int k = 0; k < 3; ++k) if (gw[k]) { g.B[n] = sc->d_h + k * hs; g.C[n] = gw[k]->w1; ++n; }
        g.groups = n;
        if (n) TRY(launch_gemm_umma_grouped(g, br.fork(0)));
    }
    if (d_x) {  // d_x (=|+=) sum_k d_h[k] W1[k]^T: one GEMM, k loop over the three heads
        GroupedGemm g;
        g.M = M; g.N = D; g.K = Dh; g.groups = 3; g.sum_groups = true; g.TB = true; g.lda = Dh; g.ldb = Dh; g.ldc = D; g.beta = accumulate_dx;
        for (int k = 0; k < 3; ++k) { g.A[k] = sc->d_h + k * hs; g.B[k] = heads[k].w1; }
        g.C[0] = d_x;
        TRY(launch_gemm_umma_grouped(g, s));
    }
    return br.join_deferrable();
}
