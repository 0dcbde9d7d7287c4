// fp32 SIMT flash-style attention (head dim 32 or 64) forward + backward: the 1e-5 parity mode.
// Reference: MultiheadAttention.call, /root/reference/ModelComponents/transformers.py:77-100.
// Layouts: qp/kp/vp are the Dense outputs [B,L,H*d] (head h = columns h*d..h*d+d-1, i.e. the
// reference's Reshape+Permute), the output is written as [B,H,Lq,d] and later re-read as
// [B,Lq,H*d] without a permute (reference line :100, SURVEY quirk Q1).
// Scores are never materialised: K/V tiles are staged in shared memory, one thread owns one query
// row (forward, dQ) or one key row (dK/dV) with its 32-wide vectors in registers.  At head dim 64 two adjacent lanes
// share a row, each holding 32 of its columns, and add their partial dot products with one shuffle: a dK/dV thread
// holding whole 64-wide rows would need 4 x 64 accumulator registers, more than a thread has.
#include <math_constants.h>
#include <cstdlib>
#include "kernels.cuh"

namespace bdetr {

constexpr int AT_COLS = 32;      // columns of a row held by one thread
constexpr int AT_THREADS = 128;  // threads per CTA (= rows per CTA at head dim 32)
constexpr int AT_TILE = 64;      // staged rows of the other operand
constexpr int AT_CHUNK = 16;
constexpr float LOG2E = 1.4426950408889634f;

__device__ __forceinline__ void load_row32(const float *p, float r[AT_COLS])
{
#pragma unroll
    for (int k = 0; k < AT_COLS / 4; ++k) {
        const float4 v = reinterpret_cast<const float4 *>(p)[k];
        r[4 * k] = v.x; r[4 * k + 1] = v.y; r[4 * k + 2] = v.z; r[4 * k + 3] = v.w;
    }
}
__device__ __forceinline__ void store_row32(float *p, const float r[AT_COLS])
{
#pragma unroll
    for (int k = 0; k < AT_COLS / 4; ++k) reinterpret_cast<float4 *>(p)[k] = make_float4(r[4 * k], r[4 * k + 1], r[4 * k + 2], r[4 * k + 3]);
}
__device__ __forceinline__ float dot32(const float a[AT_COLS], const float *sm)
{
    float s = 0.0f;
#pragma unroll
    for (int k = 0; k < AT_COLS / 4; ++k) {
        const float4 v = reinterpret_cast<const float4 *>(sm)[k];
        s = fmaf(a[4 * k], v.x, s); s = fmaf(a[4 * k + 1], v.y, s); s = fmaf(a[4 * k + 2], v.z, s); s = fmaf(a[4 * k + 3], v.w, s);
    }
    return s;
}
__device__ __forceinline__ void axpy32(float acc[AT_COLS], float a, const float *sm)
{
#pragma unroll
    for (int k = 0; k < AT_COLS / 4; ++k) {
        const float4 v = reinterpret_cast<const float4 *>(sm)[k];
        acc[4 * k] = fmaf(a, v.x, acc[4 * k]); acc[4 * k + 1] = fmaf(a, v.y, acc[4 * k + 1]);
        acc[4 * k + 2] = fmaf(a, v.z, acc[4 * k + 2]); acc[4 * k + 3] = fmaf(a, v.w, acc[4 * k + 3]);
    }
}

// sum of a row's partial dot products over the CS lanes that share the row (the same value in each of them); the
// lanes of a pair are live or idle together, so the pair's own mask is enough inside per-row branches
template <int CS>
__device__ __forceinline__ float row_sum(float s)
{
    if constexpr (CS == 2) s += __shfl_xor_sync(3u << (threadIdx.x & 30), s, 1);
    return s;
}

// stage `rows` rows of a [*, ld] matrix (HD floats each, starting at column offset already applied)
template <int HD>
__device__ __forceinline__ void stage_rows(float (*dst)[HD], const float *src, size_t ld, int rows, int valid)
{
    for (int e = threadIdx.x; e < rows * (HD / 4); e += blockDim.x) {
        const int r = e / (HD / 4), c4 = e % (HD / 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (r < valid) v = reinterpret_cast<const float4 *>(src + (size_t)r * ld)[c4];
        reinterpret_cast<float4 *>(dst[r])[c4] = v;
    }
}

// (at head dim 64 the register heuristic otherwise aims at 4 CTAs per SM, 128 registers, and spills; 0 = no minimum)
template <int HD>
__global__ void __launch_bounds__(AT_THREADS, HD == 32 ? 0 : 1)
attention_fwd_kernel(int H, int Lq, int Lk, const float *__restrict__ qp, const float *__restrict__ kp,
                     const float *__restrict__ vp, float *__restrict__ o, float *__restrict__ lse, float scale_log2, int round_out)
{
    constexpr int CS = HD / AT_COLS, RW = AT_THREADS / CS;     // lanes per row, rows per CTA
    pdl_sync();
    __shared__ __align__(16) float Ks[AT_TILE][HD];
    __shared__ __align__(16) float Vs[AT_TILE][HD];
    const int b = blockIdx.z, h = blockIdx.y, D = H * HD;
    const int i = blockIdx.x * RW + threadIdx.x / CS, col = (threadIdx.x % CS) * AT_COLS;
    const bool live = i < Lq;
    float q[AT_COLS], acc[AT_COLS];
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) { q[k] = 0.0f; acc[k] = 0.0f; }
    if (live) load_row32(qp + ((size_t)b * Lq + i) * D + h * HD + col, q);
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) q[k] *= scale_log2;        // scores in log2 units
    float m = -CUDART_INF_F, l = 0.0f;
    const float *kb = kp + (size_t)b * Lk * D + h * HD;
    const float *vb = vp + (size_t)b * Lk * D + h * HD;

    for (int k0 = 0; k0 < Lk; k0 += AT_TILE) {
        const int valid = min(AT_TILE, Lk - k0);
        __syncthreads();
        stage_rows(Ks, kb + (size_t)k0 * D, D, AT_TILE, valid);
        stage_rows(Vs, vb + (size_t)k0 * D, D, AT_TILE, valid);
        __syncthreads();
        for (int c0 = 0; c0 < valid; c0 += AT_CHUNK) {
            float s[AT_CHUNK];
            float cmax = -CUDART_INF_F;
#pragma unroll
            for (int j = 0; j < AT_CHUNK; ++j) {
                s[j] = (c0 + j < valid) ? row_sum<CS>(dot32(q, Ks[c0 + j] + col)) : -CUDART_INF_F;
                cmax = fmaxf(cmax, s[j]);
            }
            const float m_new = fmaxf(m, cmax);
            const float alpha = exp2f(m - m_new);            // m = -inf on the first chunk -> 0
            l *= alpha;
#pragma unroll
            for (int k = 0; k < AT_COLS; ++k) acc[k] *= alpha;
#pragma unroll
            for (int j = 0; j < AT_CHUNK; ++j) {
                const float p = exp2f(s[j] - m_new);          // masked -> 0
                l += p;
                axpy32(acc, p, Vs[c0 + j] + col);
            }
            m = m_new;
        }
    }
    if (live) {
        const float inv = 1.0f / l;
#pragma unroll
        for (int k = 0; k < AT_COLS; ++k) acc[k] = maybe_tf32(acc[k] * inv, round_out);
        store_row32(o + (((size_t)b * H + h) * Lq + i) * HD + col, acc);
        if (col == 0) lse[((size_t)b * H + h) * Lq + i] = m + log2f(l);     // log2 units
    }
}

// dQ: thread = query row.  Also writes delta[b,h,i] = sum_d dO*O for the dK/dV kernel.
template <int HD>
__global__ void __launch_bounds__(AT_THREADS)
attention_bwd_dq_kernel(int H, int Lq, int Lk, const float *__restrict__ qp, const float *__restrict__ kp,
                        const float *__restrict__ vp, const float *__restrict__ o, const float *__restrict__ lse,
                        const float *__restrict__ d_o, float *__restrict__ delta, float *__restrict__ d_qp,
                        float scale, float scale_log2, int round_out)
{
    constexpr int CS = HD / AT_COLS, RW = AT_THREADS / CS;     // lanes per row, rows per CTA
    pdl_sync();
    __shared__ __align__(16) float Ks[AT_TILE][HD];
    __shared__ __align__(16) float Vs[AT_TILE][HD];
    const int b = blockIdx.z, h = blockIdx.y, D = H * HD;
    const int i = blockIdx.x * RW + threadIdx.x / CS, col = (threadIdx.x % CS) * AT_COLS;
    const bool live = i < Lq;
    float q[AT_COLS], go[AT_COLS], dq[AT_COLS];
    float dl = 0.0f, my_lse = 0.0f;
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) { q[k] = 0.0f; go[k] = 0.0f; dq[k] = 0.0f; }
    if (live) {
        const size_t row = ((size_t)b * H + h) * Lq + i;
        load_row32(qp + ((size_t)b * Lq + i) * D + h * HD + col, q);
        load_row32(d_o + row * HD + col, go);
        float ov[AT_COLS];
        load_row32(o + row * HD + col, ov);
#pragma unroll
        for (int k = 0; k < AT_COLS; ++k) dl = fmaf(go[k], ov[k], dl);
        dl = row_sum<CS>(dl);
        if (col == 0) delta[row] = dl;
        my_lse = lse[row];
    }
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) q[k] *= scale_log2;
    const float *kb = kp + (size_t)b * Lk * D + h * HD;
    const float *vb = vp + (size_t)b * Lk * D + h * HD;
    for (int k0 = 0; k0 < Lk; k0 += AT_TILE) {
        const int valid = min(AT_TILE, Lk - k0);
        __syncthreads();
        stage_rows(Ks, kb + (size_t)k0 * D, D, AT_TILE, valid);
        stage_rows(Vs, vb + (size_t)k0 * D, D, AT_TILE, valid);
        __syncthreads();
        for (int j = 0; j < valid; ++j) {
            const float p = exp2f(row_sum<CS>(dot32(q, Ks[j] + col)) - my_lse);
            const float dp = row_sum<CS>(dot32(go, Vs[j] + col));
            const float ds = p * (dp - dl) * scale;
            axpy32(dq, ds, Ks[j] + col);
        }
    }
    if (live) {
#pragma unroll
        for (int k = 0; k < AT_COLS; ++k) dq[k] = maybe_tf32(dq[k], round_out);
        store_row32(d_qp + ((size_t)b * Lq + i) * D + h * HD + col, dq);
    }
}

// dK, dV: thread = key row; queries / dO / lse / delta staged in shared memory.
template <int HD>
__global__ void __launch_bounds__(AT_THREADS)
attention_bwd_dkv_kernel(int H, int Lq, int Lk, const float *__restrict__ qp, const float *__restrict__ kp,
                         const float *__restrict__ vp, const float *__restrict__ lse, const float *__restrict__ d_o,
                         const float *__restrict__ delta, float *__restrict__ d_kp, float *__restrict__ d_vp,
                         float scale, float scale_log2, int round_out)
{
    constexpr int CS = HD / AT_COLS, RW = AT_THREADS / CS;
    pdl_sync();
    __shared__ __align__(16) float Qs[AT_TILE][HD];
    __shared__ __align__(16) float Gs[AT_TILE][HD];
    __shared__ float Ls[AT_TILE], Ds[AT_TILE];
    const int b = blockIdx.z, h = blockIdx.y, D = H * HD;
    const int j = blockIdx.x * RW + threadIdx.x / CS, col = (threadIdx.x % CS) * AT_COLS;
    const bool live = j < Lk;
    float kr[AT_COLS], vr[AT_COLS], dk[AT_COLS], dv[AT_COLS];
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) { kr[k] = 0.0f; vr[k] = 0.0f; dk[k] = 0.0f; dv[k] = 0.0f; }
    if (live) {
        load_row32(kp + ((size_t)b * Lk + j) * D + h * HD + col, kr);
        load_row32(vp + ((size_t)b * Lk + j) * D + h * HD + col, vr);
    }
#pragma unroll
    for (int k = 0; k < AT_COLS; ++k) kr[k] *= scale_log2;      // so that dot(kr, q) is the log2-unit score
    const float *qb = qp + (size_t)b * Lq * D + h * HD;
    const size_t rowbase = ((size_t)b * H + h) * Lq;
    for (int i0 = 0; i0 < Lq; i0 += AT_TILE) {
        const int valid = min(AT_TILE, Lq - i0);
        __syncthreads();
        stage_rows(Qs, qb + (size_t)i0 * D, D, AT_TILE, valid);
        stage_rows(Gs, d_o + (rowbase + i0) * HD, HD, AT_TILE, valid);
        for (int e = threadIdx.x; e < AT_TILE; e += blockDim.x) {
            Ls[e] = e < valid ? lse[rowbase + i0 + e] : 0.0f;
            Ds[e] = e < valid ? delta[rowbase + i0 + e] : 0.0f;
        }
        __syncthreads();
        for (int i = 0; i < valid; ++i) {
            const float p = exp2f(row_sum<CS>(dot32(kr, Qs[i] + col)) - Ls[i]);
            axpy32(dv, p, Gs[i] + col);
            const float dp = row_sum<CS>(dot32(vr, Gs[i] + col));
            const float ds = p * (dp - Ds[i]) * scale;
            axpy32(dk, ds, Qs[i] + col);
        }
    }
    if (live) {
#pragma unroll
        for (int k = 0; k < AT_COLS; ++k) { dk[k] = maybe_tf32(dk[k], round_out); dv[k] = maybe_tf32(dv[k], round_out); }
        store_row32(d_kp + ((size_t)b * Lk + j) * D + h * HD + col, dk);
        store_row32(d_vp + ((size_t)b * Lk + j) * D + h * HD + col, dv);
    }
}

int g_force_attention_kernel = 0;       // 0 auto, 1 one tile per CTA, 2 multi-stream (bdetr_debug_force_attention_kernel)

namespace {

template <int HD>
int launch_fwd_simt(int B, int H, int Lq, int Lk, const float *qp, const float *kp, const float *vp, float *o, float *lse,
                     int round_out, cudaStream_t s)
{
    const float scale = 1.0f / sqrtf((float)HD);
    dim3 grid(ceil_div(Lq, AT_THREADS * AT_COLS / HD), H, B);
    launch_k(attention_fwd_kernel<HD>, grid, AT_THREADS, 0, s, H, Lq, Lk, qp, kp, vp, o, lse, scale * LOG2E, round_out);
    BDETR_CHECK_LAUNCH("attention_fwd_kernel");
    return BDETR_OK;
}

template <int HD>
int launch_bwd_simt(int B, int H, int Lq, int Lk, const float *qp, const float *kp, const float *vp, const float *o,
                     const float *lse, const float *d_o, float *delta, float *d_qp, float *d_kp, float *d_vp, int round_out,
                     cudaStream_t s)
{
    const float scale = 1.0f / sqrtf((float)HD);
    dim3 gq(ceil_div(Lq, AT_THREADS * AT_COLS / HD), H, B);
    launch_k(attention_bwd_dq_kernel<HD>, gq, AT_THREADS, 0, s, H, Lq, Lk, qp, kp, vp, o, lse, d_o, delta, d_qp, scale, scale * LOG2E, round_out);
    BDETR_CHECK_LAUNCH("attention_bwd_dq_kernel");
    dim3 gk(ceil_div(Lk, AT_THREADS * AT_COLS / HD), H, B);
    launch_k(attention_bwd_dkv_kernel<HD>, gk, AT_THREADS, 0, s, H, Lq, Lk, qp, kp, vp, lse, d_o, delta, d_kp, d_vp, scale, scale * LOG2E, round_out);
    BDETR_CHECK_LAUNCH("attention_bwd_dkv_kernel");
    return BDETR_OK;
}

}  // namespace

int launch_attention_fwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                         float *o, float *lse, int round_out, cudaStream_t s)
{
    BDETR_REQUIRE(d == 32 || d == 64, BDETR_E_UNSUPPORTED, "head dim must be 32 or 64 (D/H)");
    BDETR_REQUIRE(B > 0 && H > 0 && Lq > 0 && Lk > 0, BDETR_E_BAD_SHAPE, "bad attention shape");
    if (current_mode() == BDETR_MODE_TF32 && attention_umma_eligible(B, H, Lq, Lk, d, qp, kp, vp)) {
        // long sequences at head dim 32: three query tiles per CTA against a shared K/V ring (attention_umma_ms.cu, which
        // refuses other head dims when forced)
        const int force = g_force_attention_kernel;
        if (force == 2 || (force >= 20 && force <= 28) || (force == 0 && d == 32 && attention_umma_ms_eligible(B, H, Lq, Lk)))
            return launch_attention_fwd_umma_ms(B, H, Lq, Lk, d, qp, kp, vp, o, lse, round_out, s);
        return launch_attention_fwd_umma(B, H, Lq, Lk, d, qp, kp, vp, o, lse, round_out, s);
    }
    return d == 64 ? launch_fwd_simt<64>(B, H, Lq, Lk, qp, kp, vp, o, lse, round_out, s)
                   : launch_fwd_simt<32>(B, H, Lq, Lk, qp, kp, vp, o, lse, round_out, s);
}

int launch_attention_bwd(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                         const float *o, const float *lse, const float *d_o, float *delta,
                         float *d_qp, float *d_kp, float *d_vp, int round_out, cudaStream_t s)
{
    BDETR_REQUIRE(d == 32 || d == 64, BDETR_E_UNSUPPORTED, "head dim must be 32 or 64 (D/H)");
    if (current_mode() == BDETR_MODE_TF32 && attention_bwd_umma_eligible(B, H, Lq, Lk, d, qp, kp, vp, d_o))
        return launch_attention_bwd_umma(B, H, Lq, Lk, d, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, round_out, s);
    return d == 64 ? launch_bwd_simt<64>(B, H, Lq, Lk, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, round_out, s)
                   : launch_bwd_simt<32>(B, H, Lq, Lk, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, round_out, s);
}

}  // namespace bdetr
