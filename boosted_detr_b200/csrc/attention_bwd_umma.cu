// Flash-attention backward on tcgen05 (head dim 32 or 64, TF32 operands, fp32 accumulation in TMEM).
// Two kernels, no atomics, scores recomputed from q/k and the forward's log-sum-exp (log2 units):
//
//   attention_bwd_dq_umma_kernel   CTA = 128 query rows; loop over 64-key tiles
//        S  = Q Kt, dP = dO Vt                       (SS MMAs, all operands K-major)           -> TMEM
//        dS = P o (dP - delta)                        one thread per query row (lse/delta are row scalars),
//                                                     written over S in TMEM
//        dQ += dS K                                   (A = dS from TMEM, B = K as MN-major operand)
//
//   attention_bwd_dkv_umma_kernel  CTA = 128 key rows; loop over 64-query tiles, scores TRANSPOSED so that
//        St = K Qt, dPt = V dOt                       P^T / dS^T land as [key lanes x query columns] in TMEM,
//        Pt, dSt                                      one thread per key row (lse/delta per column from smem)
//        dV += Pt dO,  dK += dSt Q                    (A from TMEM, B = dO / Q as MN-major operands)
//
// 1/sqrt(d) is folded into the dQ / dK epilogues.  P and dS are masked to tf32 precision before they are handed
// to the tensor cores.  At d = 32 two CTAs per SM (256 TMEM columns, <= 96 KB shared memory each).  At d = 64 every
// tile is two 32-column (128-byte) swizzle boxes side by side, as in attention_umma.cu: the K-major MMAs take 8 k-steps
// through both, the MN-major B operands are two 32-column atoms.  TMEM: dQ uses S 64 + dP 64 + dQ 64 columns, dK/dV
// S 64 + dP 64 + dK 64 + dV 64 = all 256; shared memory is 160 KB (dQ) and 192 KB (dK/dV): one CTA per SM.
// Reference: the gradient of MultiheadAttention.call, /root/reference/ModelComponents/transformers.py:77-100.
#include <math_constants.h>
#include "umma.cuh"

namespace bdetr {

constexpr int FB_ROWS = 128;                 // rows owned by a CTA (queries in dQ, keys in dK/dV)
constexpr int FB_T = 64;                     // looped tile (keys in dQ, queries in dK/dV)
constexpr int FB_THREADS = 192;
constexpr uint32_t FB_BIG_BOX = FB_ROWS * 32 * 4;     // 16 KB: one 128-byte-wide swizzle box of a FB_ROWS-row tile
constexpr uint32_t FB_SMALL_BOX = FB_T * 32 * 4;      // 8 KB: the same for a FB_T-row tile
constexpr uint32_t FB_TMEM = 256;
constexpr uint32_t TF32_MASK = 0xFFFFE000u;

__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// ---------------------------------------------------------------------------------------------------------
// dQ
// ---------------------------------------------------------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(FB_THREADS, HD == 32 ? 2 : 1)
attention_bwd_dq_umma_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                             const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                             const __grid_constant__ CUtensorMap map_k_mn, int H, int Lq, int Lk,
                             const float *__restrict__ o, const float *__restrict__ d_o, const float *__restrict__ lse,
                             float *__restrict__ delta, float *__restrict__ d_qp, float scale, float scale_log2, int round_out)
{
    constexpr uint32_t FB_BIG = FB_ROWS * HD * 4, FB_SMALL = FB_T * HD * 4;        // tiles of HD / 32 boxes each
    constexpr int NB = HD / 32;
    constexpr uint32_t mn_lbo = NB == 1 ? 4096 : FB_SMALL_BOX;                   // MN-major B: 32-column atoms (one at d = 32)
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *smem_q = smem, *smem_do = smem + FB_BIG;
    uint8_t *stage0 = smem + 2 * FB_BIG;                                 // [2][K_sw | V_sw | K_mn]
    uint64_t *bars = reinterpret_cast<uint64_t *>(stage0 + 2 * 3 * FB_SMALL);
    uint64_t *qdo_full = bars, *kv_full = bars + 1, *kv_empty = bars + 3, *sd_full = bars + 5, *ds_full = bars + 6, *dq_full = bars + 7;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * FB_ROWS;
    const int ntiles = (Lk + FB_T - 1) / FB_T;
    const int D = H * HD;

    if (threadIdx.x == 0) {
        mbar_init(qdo_full, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
        mbar_init(sd_full, 1); mbar_init(ds_full, 128); mbar_init(dq_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, FB_TMEM);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // PDL: dependents are released only after this CTA owns its TMEM columns (a dependent that grabbed TMEM first while
    // blocked in griddepcontrol.wait could starve a late CTA of this grid); global data is touched below the wait.
    pdl_sync();
    constexpr uint32_t COL_S = 0, COL_DP = 64, COL_DQ = 128;

    // warps 0 / 1 walk their loops warp-convergent and only the issuing instructions are predicated on one elected
    // lane (see elect_one in umma.cuh): descriptors stay in uniform registers.
    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(qdo_full, 2 * FB_BIG);
#pragma unroll
            for (int c = 0; c < NB; ++c) {
                tma_load_2d(smem_q + c * FB_BIG_BOX, &map_q, h * HD + c * 32, b * Lq + q0, qdo_full);
                tma_load_2d(smem_do + c * FB_BIG_BOX, &map_do, c * 32, (b * H + h) * Lq + q0, qdo_full);
            }
        }
        __syncwarp();
        for (int t = 0; t < ntiles; ++t) {
            const int s = t & 1;
            if (t >= 2) mbar_wait(&kv_empty[s], ((t >> 1) - 1) & 1);
            uint8_t *st = stage0 + s * 3 * FB_SMALL;
            const int krow = b * Lk + t * FB_T;
            if (elect_one()) {
                mbar_expect_tx(&kv_full[s], 3 * FB_SMALL);
#pragma unroll
                for (int c = 0; c < NB; ++c) {
                    tma_load_2d(st + c * FB_SMALL_BOX, &map_k, h * HD + c * 32, krow, &kv_full[s]);
                    tma_load_2d(st + FB_SMALL + c * FB_SMALL_BOX, &map_v, h * HD + c * 32, krow, &kv_full[s]);
                    tma_load_2d(st + 2 * FB_SMALL + c * FB_SMALL_BOX, &map_k_mn, h * HD + c * 32, krow, &kv_full[s]);
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc_s = make_idesc_tf32(FB_ROWS, FB_T, 0, 0);
        constexpr uint32_t idesc_q = make_idesc_tf32(FB_ROWS, HD, 0, 1);
        mbar_wait(qdo_full, 0);
        const uint32_t q_base = smem_u32(smem_q), do_base = smem_u32(smem_do);
        for (int t = 0; t < ntiles; ++t) {
            const int s = t & 1;
            mbar_wait(&kv_full[s], (t >> 1) & 1);
            tc_fence_after();
            const uint32_t k_base = smem_u32(stage0 + s * 3 * FB_SMALL), v_base = k_base + FB_SMALL, kmn_base = k_base + 2 * FB_SMALL;
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < HD / 8; ++j)         // k-step j: box j / 4 of each tile, 32-byte column j % 4 of it
                    umma_tf32(tmem_base + COL_S, make_smem_desc(q_base + (j / 4) * FB_BIG_BOX + (j % 4) * 32, 16, 1024, 2),
                              make_smem_desc(k_base + (j / 4) * FB_SMALL_BOX + (j % 4) * 32, 16, 1024, 2), idesc_s, j != 0);
#pragma unroll
                for (int j = 0; j < HD / 8; ++j)
                    umma_tf32(tmem_base + COL_DP, make_smem_desc(do_base + (j / 4) * FB_BIG_BOX + (j % 4) * 32, 16, 1024, 2),
                              make_smem_desc(v_base + (j / 4) * FB_SMALL_BOX + (j % 4) * 32, 16, 1024, 2), idesc_s, j != 0);
                umma_commit(sd_full);
            }
            __syncwarp();
            mbar_wait(ds_full, t & 1);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < FB_T / 8; ++j)
                    umma_tf32_ts(tmem_base + COL_DQ, tmem_base + COL_S + j * 8, make_smem_desc(kmn_base + j * 1024, mn_lbo, 512, 1), idesc_q, (t | j) != 0);
                umma_commit(&kv_empty[s]);
                if (t == ntiles - 1) umma_commit(dq_full);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3;
        const int row = q0 + q * 32 + lane;
        const bool live = row < Lq;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        const size_t orow = ((size_t)b * H + h) * Lq + row;
        // delta = sum_d dO * O for this row (also handed to the dK/dV kernel)
        float dl = 0.0f, lse_r = 0.0f;
        if (live) {
#pragma unroll
            for (int i = 0; i < HD; i += 4) {
                const float4 g = *reinterpret_cast<const float4 *>(d_o + orow * HD + i);
                const float4 ov = *reinterpret_cast<const float4 *>(o + orow * HD + i);
                dl = fmaf(g.x, ov.x, dl); dl = fmaf(g.y, ov.y, dl); dl = fmaf(g.z, ov.z, dl); dl = fmaf(g.w, ov.w, dl);
            }
            delta[orow] = dl;
            lse_r = lse[orow];
        }
        for (int t = 0; t < ntiles; ++t) {
            const int valid = min(FB_T, Lk - t * FB_T);
            mbar_wait(sd_full, t & 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < FB_T / 32; ++c) {
                uint32_t rs[32], rp[32];
                tmem_ld32_issue(lane_addr + COL_S + c * 32, rs);
                tmem_ld32_issue(lane_addr + COL_DP + c * 32, rp);
                tmem_ld32_wait(rs);
                tmem_ld32_wait(rp);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float p = ex2_approx(fmaf(__uint_as_float(rs[i]), scale_log2, -lse_r));
                    uint32_t ds = __float_as_uint(p * (__uint_as_float(rp[i]) - dl)) & TF32_MASK;
                    if (c * 32 + i >= valid) ds = 0u;
                    rs[i] = ds;
                }
                tmem_st32_u(lane_addr + COL_S + c * 32, rs);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(ds_full);
        }
        mbar_wait(dq_full, 0);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < NB; ++c) {
            float acc[32];
            tmem_ld32(lane_addr + COL_DQ + c * 32, acc);
            if (live) {
                float *dst = d_qp + ((size_t)b * Lq + row) * D + h * HD + c * 32;
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    float4 w = make_float4(acc[i] * scale, acc[i + 1] * scale, acc[i + 2] * scale, acc[i + 3] * scale);
                    if (round_out) { w.x = tf32_rn(w.x); w.y = tf32_rn(w.y); w.z = tf32_rn(w.z); w.w = tf32_rn(w.w); }
                    *reinterpret_cast<float4 *>(dst + i) = w;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, FB_TMEM);
}

// ---------------------------------------------------------------------------------------------------------
// dK, dV
// ---------------------------------------------------------------------------------------------------------
template <int HD>
__global__ void __launch_bounds__(FB_THREADS, HD == 32 ? 2 : 1)
attention_bwd_dkv_umma_kernel(const __grid_constant__ CUtensorMap map_k, const __grid_constant__ CUtensorMap map_v,
                              const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_do,
                              const __grid_constant__ CUtensorMap map_q_mn, const __grid_constant__ CUtensorMap map_do_mn,
                              int H, int Lq, int Lk, const float *__restrict__ lse, const float *__restrict__ delta,
                              float *__restrict__ d_kp, float *__restrict__ d_vp, float scale, float scale_log2, int round_out)
{
    constexpr uint32_t FB_BIG = FB_ROWS * HD * 4, FB_SMALL = FB_T * HD * 4;        // tiles of HD / 32 boxes each
    constexpr int NB = HD / 32;
    constexpr uint32_t mn_lbo = NB == 1 ? 4096 : FB_SMALL_BOX;                   // MN-major B: 32-column atoms (one at d = 32)
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *smem_k = smem, *smem_v = smem + FB_BIG;
    uint8_t *stage0 = smem + 2 * FB_BIG;                                 // [2][Q_sw | dO_sw | Q_mn | dO_mn]
    float2 *ld_s = reinterpret_cast<float2 *>(stage0 + 2 * 4 * FB_SMALL);         // [2][64] (lse, delta) per query column
    uint64_t *bars = reinterpret_cast<uint64_t *>(ld_s + 2 * FB_T);
    uint64_t *kv_full = bars, *q_full = bars + 1, *q_empty = bars + 3, *sd_full = bars + 5, *pd_full = bars + 6, *acc_full = bars + 7;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 8);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.z, h = blockIdx.y, k0 = blockIdx.x * FB_ROWS;
    const int ntiles = (Lq + FB_T - 1) / FB_T;
    const int D = H * HD;

    if (threadIdx.x == 0) {
        mbar_init(kv_full, 1);
        for (int s = 0; s < 2; ++s) { mbar_init(&q_full[s], 1); mbar_init(&q_empty[s], 1); }
        mbar_init(sd_full, 1); mbar_init(pd_full, 128); mbar_init(acc_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, FB_TMEM);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // PDL: dependents are released only after this CTA owns its TMEM columns (a dependent that grabbed TMEM first while
    // blocked in griddepcontrol.wait could starve a late CTA of this grid); global data is touched below the wait.
    pdl_sync();
    constexpr uint32_t COL_S = 0, COL_DP = 64, COL_DK = 128, COL_DV = 128 + HD;
    const int orow0 = (b * H + h) * Lq;

    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(kv_full, 2 * FB_BIG);
#pragma unroll
            for (int c = 0; c < NB; ++c) {
                tma_load_2d(smem_k + c * FB_BIG_BOX, &map_k, h * HD + c * 32, b * Lk + k0, kv_full);
                tma_load_2d(smem_v + c * FB_BIG_BOX, &map_v, h * HD + c * 32, b * Lk + k0, kv_full);
            }
        }
        __syncwarp();
        for (int t = 0; t < ntiles; ++t) {
            const int s = t & 1;
            if (t >= 2) mbar_wait(&q_empty[s], ((t >> 1) - 1) & 1);
            uint8_t *st = stage0 + s * 4 * FB_SMALL;
            const int qrow = b * Lq + t * FB_T, gorow = orow0 + t * FB_T;
            if (elect_one()) {
                mbar_expect_tx(&q_full[s], 4 * FB_SMALL);
#pragma unroll
                for (int c = 0; c < NB; ++c) {
                    tma_load_2d(st + c * FB_SMALL_BOX, &map_q, h * HD + c * 32, qrow, &q_full[s]);
                    tma_load_2d(st + FB_SMALL + c * FB_SMALL_BOX, &map_do, c * 32, gorow, &q_full[s]);
                    tma_load_2d(st + 2 * FB_SMALL + c * FB_SMALL_BOX, &map_q_mn, h * HD + c * 32, qrow, &q_full[s]);
                    tma_load_2d(st + 3 * FB_SMALL + c * FB_SMALL_BOX, &map_do_mn, c * 32, gorow, &q_full[s]);
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc_s = make_idesc_tf32(FB_ROWS, FB_T, 0, 0);
        constexpr uint32_t idesc_a = make_idesc_tf32(FB_ROWS, HD, 0, 1);
        mbar_wait(kv_full, 0);
        const uint32_t k_base = smem_u32(smem_k), v_base = smem_u32(smem_v);
        for (int t = 0; t < ntiles; ++t) {
            const int s = t & 1;
            mbar_wait(&q_full[s], (t >> 1) & 1);
            tc_fence_after();
            const uint32_t qsw = smem_u32(stage0 + s * 4 * FB_SMALL), dosw = qsw + FB_SMALL, qmn = qsw + 2 * FB_SMALL, domn = qsw + 3 * FB_SMALL;
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < HD / 8; ++j)
                    umma_tf32(tmem_base + COL_S, make_smem_desc(k_base + (j / 4) * FB_BIG_BOX + (j % 4) * 32, 16, 1024, 2),
                              make_smem_desc(qsw + (j / 4) * FB_SMALL_BOX + (j % 4) * 32, 16, 1024, 2), idesc_s, j != 0);
#pragma unroll
                for (int j = 0; j < HD / 8; ++j)
                    umma_tf32(tmem_base + COL_DP, make_smem_desc(v_base + (j / 4) * FB_BIG_BOX + (j % 4) * 32, 16, 1024, 2),
                              make_smem_desc(dosw + (j / 4) * FB_SMALL_BOX + (j % 4) * 32, 16, 1024, 2), idesc_s, j != 0);
                umma_commit(sd_full);
            }
            __syncwarp();
            mbar_wait(pd_full, t & 1);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < FB_T / 8; ++j)
                    umma_tf32_ts(tmem_base + COL_DV, tmem_base + COL_S + j * 8, make_smem_desc(domn + j * 1024, mn_lbo, 512, 1), idesc_a, (t | j) != 0);
#pragma unroll
                for (int j = 0; j < FB_T / 8; ++j)
                    umma_tf32_ts(tmem_base + COL_DK, tmem_base + COL_DP + j * 8, make_smem_desc(qmn + j * 1024, mn_lbo, 512, 1), idesc_a, (t | j) != 0);
                umma_commit(&q_empty[s]);
                if (t == ntiles - 1) umma_commit(acc_full);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3;
        const int ct = threadIdx.x - 64;                 // 0..127
        const int krow = k0 + q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        for (int t = 0; t < ntiles; ++t) {
            const int valid = min(FB_T, Lq - t * FB_T);
            float2 *ld = ld_s + (t & 1) * FB_T;
            if (ct < FB_T) {
                const int qi = t * FB_T + ct;
                ld[ct] = qi < Lq ? make_float2(lse[orow0 + qi], delta[orow0 + qi]) : make_float2(0.0f, 0.0f);
            }
            named_bar_sync(1, 128);
            mbar_wait(sd_full, t & 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < FB_T / 32; ++c) {
                uint32_t rs[32], rp[32];
                tmem_ld32_issue(lane_addr + COL_S + c * 32, rs);
                tmem_ld32_issue(lane_addr + COL_DP + c * 32, rp);
                tmem_ld32_wait(rs);
                tmem_ld32_wait(rp);
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                    const float2 lv = ld[c * 32 + i];
                    const float p = ex2_approx(fmaf(__uint_as_float(rs[i]), scale_log2, -lv.x));
                    uint32_t pb = __float_as_uint(p) & TF32_MASK;
                    uint32_t ds = __float_as_uint(p * (__uint_as_float(rp[i]) - lv.y)) & TF32_MASK;
                    if (c * 32 + i >= valid) { pb = 0u; ds = 0u; }
                    rs[i] = pb;
                    rp[i] = ds;
                }
                tmem_st32_u(lane_addr + COL_S + c * 32, rs);
                tmem_st32_u(lane_addr + COL_DP + c * 32, rp);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(pd_full);
        }
        mbar_wait(acc_full, 0);
        tc_fence_after();
#pragma unroll
        for (int c = 0; c < NB; ++c) {
            float acc[32];
            tmem_ld32(lane_addr + COL_DK + c * 32, acc);
            if (krow < Lk) {
                float *dst = d_kp + ((size_t)b * Lk + krow) * D + h * HD + c * 32;
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    float4 w = make_float4(acc[i] * scale, acc[i + 1] * scale, acc[i + 2] * scale, acc[i + 3] * scale);
                    if (round_out) { w.x = tf32_rn(w.x); w.y = tf32_rn(w.y); w.z = tf32_rn(w.z); w.w = tf32_rn(w.w); }
                    *reinterpret_cast<float4 *>(dst + i) = w;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < NB; ++c) {
            float acc[32];
            tmem_ld32(lane_addr + COL_DV + c * 32, acc);
            if (krow < Lk) {
                float *dst = d_vp + ((size_t)b * Lk + krow) * D + h * HD + c * 32;
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    float4 w = make_float4(acc[i], acc[i + 1], acc[i + 2], acc[i + 3]);
                    if (round_out) { w.x = tf32_rn(w.x); w.y = tf32_rn(w.y); w.z = tf32_rn(w.z); w.w = tf32_rn(w.w); }
                    *reinterpret_cast<float4 *>(dst + i) = w;
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, FB_TMEM);
}

bool attention_bwd_umma_eligible(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                                 const float *d_o)
{
    auto al = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return (d == 32 || d == 64) && al(qp) && al(kp) && al(vp) && al(d_o) && B >= 1 && Lq >= 1 && Lk >= 1;
}

namespace {

template <int HD>
int launch_bwd_umma(int B, int H, int Lq, int Lk, const float *qp, const float *kp, const float *vp, const float *o,
                    const float *lse, const float *d_o, float *delta, float *d_qp, float *d_kp, float *d_vp, int round_out,
                    cudaStream_t s)
{
    const int D = H * HD;
    const long long rq = (long long)B * Lq, rk = (long long)B * Lk, ro = (long long)B * H * Lq;
    // every box is 32 columns (128 bytes, the widest SWIZZLE_128B box); a d = 64 tile is two of them
    CUtensorMap q128, do128, k64, v64, k64mn, k128, v128, q64, do64, q64mn, do64mn;
    bool ok = encode_tensor_map_2d(&q128, qp, rq, D, D, 32, FB_ROWS, false);
    ok = ok && encode_tensor_map_2d(&do128, d_o, ro, HD, HD, 32, FB_ROWS, false);
    ok = ok && encode_tensor_map_2d(&k64, kp, rk, D, D, 32, FB_T, false);
    ok = ok && encode_tensor_map_2d(&v64, vp, rk, D, D, 32, FB_T, false);
    ok = ok && encode_tensor_map_2d(&k64mn, kp, rk, D, D, 32, FB_T, true);
    ok = ok && encode_tensor_map_2d(&k128, kp, rk, D, D, 32, FB_ROWS, false);
    ok = ok && encode_tensor_map_2d(&v128, vp, rk, D, D, 32, FB_ROWS, false);
    ok = ok && encode_tensor_map_2d(&q64, qp, rq, D, D, 32, FB_T, false);
    ok = ok && encode_tensor_map_2d(&do64, d_o, ro, HD, HD, 32, FB_T, false);
    ok = ok && encode_tensor_map_2d(&q64mn, qp, rq, D, D, 32, FB_T, true);
    ok = ok && encode_tensor_map_2d(&do64mn, d_o, ro, HD, HD, 32, FB_T, true);
    BDETR_REQUIRE(ok, BDETR_E_CUDA, "cuTensorMapEncodeTiled failed");
    const float scale = 1.0f / sqrtf((float)HD), scale_log2 = scale * 1.4426950408889634f;
    constexpr size_t big = FB_ROWS * HD * 4, small = FB_T * HD * 4;
    const size_t smem_dq = 2 * big + 2 * 3 * small + 16 * 8 + 1024;
    const size_t smem_dkv = 2 * big + 2 * 4 * small + 2 * FB_T * 8 + 16 * 8 + 1024;
    static bool optin = false;
    if (!optin) {
        BDETR_CUDA(cudaFuncSetAttribute(attention_bwd_dq_umma_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_dq));
        BDETR_CUDA(cudaFuncSetAttribute(attention_bwd_dkv_umma_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_dkv));
        optin = true;
    }
    // (dQ and dK/dV back to back on one stream: running them side by side -- delta from a kernel of its own -- was measured
    // and dropped, 2.55 -> 2.69 ms per step: two 512-CTA kernels at once thrash the SM slots the backward is bound by)
    dim3 gq(ceil_div(Lq, FB_ROWS), H, B);
    launch_k(attention_bwd_dq_umma_kernel<HD>, gq, FB_THREADS, smem_dq, s, q128, do128, k64, v64, k64mn, H, Lq, Lk, o, d_o, lse, delta,
             d_qp, scale, scale_log2, round_out);
    BDETR_CHECK_LAUNCH("attention_bwd_dq_umma_kernel");
    dim3 gk(ceil_div(Lk, FB_ROWS), H, B);
    launch_k(attention_bwd_dkv_umma_kernel<HD>, gk, FB_THREADS, smem_dkv, s, k128, v128, q64, do64, q64mn, do64mn, H, Lq, Lk, lse,
             delta, d_kp, d_vp, scale, scale_log2, round_out);
    BDETR_CHECK_LAUNCH("attention_bwd_dkv_umma_kernel");
    return BDETR_OK;
}

}  // namespace

int launch_attention_bwd_umma(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                              const float *o, const float *lse, const float *d_o, float *delta,
                              float *d_qp, float *d_kp, float *d_vp, int round_out, cudaStream_t s)
{
    BDETR_REQUIRE(d == 32 || d == 64, BDETR_E_UNSUPPORTED, "head dim must be 32 or 64 (D/H)");
    return d == 64 ? launch_bwd_umma<64>(B, H, Lq, Lk, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, round_out, s)
                   : launch_bwd_umma<32>(B, H, Lq, Lk, qp, kp, vp, o, lse, d_o, delta, d_qp, d_kp, d_vp, round_out, s);
}

}  // namespace bdetr
