// Flash-style attention forward on the 5th-generation tensor cores (head dim 32 or 64, TF32 operands, fp32 state).
// Reference: MultiheadAttention.call, /root/reference/ModelComponents/transformers.py:77-100 — the scores
// [B,H,Lq,Lk] are never materialised in HBM.
//
// CTA = (128 query rows, head h, image b); 192 threads:
//   warp 0      TMA producer: Q tile once, then a 2-stage ring of (K tile, V tile) — 128 keys each
//   warp 1      TMEM allocator + single-thread tcgen05.mma issuer
//                   S[128x128]  = Q Kt        A, B K-major from shared memory (SWIZZLE_128B)      -> TMEM cols 0..127
//                   Ot[128xd]   = P V         A = P from TMEM, B = V MN-major (SWIZZLE_128B_BASE32B) -> TMEM cols 128..128+d-1
//   warps 2..5  softmax: one thread per query row (TMEM lane).  Two passes over the S row in TMEM (row max,
//               then exp2 / row sum), P written back in place over S (masked to tf32 precision, and the row sum
//               taken over the masked values, so the MMA's operand truncation is exact and cancels in the
//               normalisation), running (m, l, o[d]) in registers: o = o*alpha + Ot after each tile.
// Keeping O in registers makes the online-softmax rescale free (no TMEM correction pass).  At d = 32 two CTAs per SM
// (80 KB shared memory, 256 TMEM columns each) overlap one CTA's softmax with the other's MMAs.  At d = 64 a 256-byte
// row is two 128-byte swizzle boxes: every Q, K and V tile is two 32-column boxes side by side, S = Q Kt takes 8 k-steps
// through both, and PV reads V as two 32-column MN-major atoms (the gemm_umma.cu layout).  The tiles stay 128 keys, so
// a CTA holds 160 KB of shared memory and runs alone on its SM; Ot uses 64 of the 256 TMEM columns.
// Output layout [B,H,Lq,d] (quirk Q1), log-sum-exp in log2 units like the SIMT kernel (shared backward).
#include <math_constants.h>
#include "umma.cuh"

namespace bdetr {

constexpr int FA_BM = 128;      // query rows per CTA
constexpr int FA_KT = 128;      // keys per tile
constexpr int FA_THREADS = 192;
constexpr int FA_STAGES = 2;
constexpr uint32_t FA_BOX_BYTES = FA_KT * 32 * 4;          // 16 KB: 128 rows x 32 columns, one 128-byte swizzle box
constexpr uint32_t FA_TMEM_COLS = 256;
constexpr uint32_t FA_O_COL = 128;

template <int HD>
__global__ void __launch_bounds__(FA_THREADS, HD == 32 ? 2 : 1)
attention_fwd_umma_kernel(const __grid_constant__ CUtensorMap map_q, const __grid_constant__ CUtensorMap map_k,
                          const __grid_constant__ CUtensorMap map_v, int H, int Lq, int Lk,
                          float *__restrict__ o, float *__restrict__ lse, float scale_log2, int round_out)
{
    constexpr uint32_t FA_TILE_BYTES = FA_KT * HD * 4;     // Q, K and V tiles: HD / 32 boxes side by side
    constexpr int NB = HD / 32;
    extern __shared__ uint8_t smem_raw[];
    uint8_t *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    uint8_t *smem_q = smem;
    uint8_t *smem_k = smem_q + FA_TILE_BYTES;
    uint8_t *smem_v = smem_k + FA_STAGES * FA_TILE_BYTES;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_v + FA_STAGES * FA_TILE_BYTES);
    uint64_t *q_full = bars, *kv_full = bars + 1, *kv_empty = kv_full + FA_STAGES;
    uint64_t *s_full = kv_empty + FA_STAGES, *p_full = s_full + 1, *o_full = p_full + 1;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(o_full + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * FA_BM;
    const int ntiles = (Lk + FA_KT - 1) / FA_KT;

    if (threadIdx.x == 0) {
        mbar_init(q_full, 1);
        for (int s = 0; s < FA_STAGES; ++s) { mbar_init(&kv_full[s], 1); mbar_init(&kv_empty[s], 1); }
        mbar_init(s_full, 1);
        mbar_init(p_full, 128);
        mbar_init(o_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) tmem_alloc(tmem_slot, FA_TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // PDL: dependents are released only after this CTA owns its TMEM columns (a dependent that grabbed TMEM first while
    // blocked in griddepcontrol.wait could starve a late CTA of this grid); global data is touched below the wait.
    pdl_sync();

    // warps 0 / 1 walk their loops warp-convergent; only the issuing instructions are predicated on one elected lane
    // (see elect_one in umma.cuh): descriptors stay in uniform registers.
    if (warp == 0) {
        if (elect_one()) {
            mbar_expect_tx(q_full, FA_TILE_BYTES);
#pragma unroll
            for (int c = 0; c < NB; ++c) tma_load_2d(smem_q + c * FA_BOX_BYTES, &map_q, h * HD + c * 32, b * Lq + q0, q_full);
        }
        __syncwarp();
        for (int t = 0; t < ntiles; ++t) {
            const int s = t % FA_STAGES;
            if (t >= FA_STAGES) mbar_wait(&kv_empty[s], ((t / FA_STAGES) - 1) & 1);
            if (elect_one()) {
                mbar_expect_tx(&kv_full[s], 2 * FA_TILE_BYTES);
#pragma unroll
                for (int c = 0; c < NB; ++c) {
                    tma_load_2d(smem_k + s * FA_TILE_BYTES + c * FA_BOX_BYTES, &map_k, h * HD + c * 32, b * Lk + t * FA_KT, &kv_full[s]);
                    tma_load_2d(smem_v + s * FA_TILE_BYTES + c * FA_BOX_BYTES, &map_v, h * HD + c * 32, b * Lk + t * FA_KT, &kv_full[s]);
                }
            }
            __syncwarp();
        }
    } else if (warp == 1) {
        constexpr uint32_t idesc_s = make_idesc_tf32(FA_BM, FA_KT, 0, 0);      // both K-major
        constexpr uint32_t idesc_o = make_idesc_tf32(FA_BM, HD, 0, 1);         // A from TMEM, B (V) MN-major
        constexpr uint32_t v_lbo = NB == 1 ? 4096 : FA_BOX_BYTES;              // V's 32-column atoms (one at d = 32)
        mbar_wait(q_full, 0);
        const uint32_t q_base = smem_u32(smem_q);
        for (int t = 0; t < ntiles; ++t) {
            const int s = t % FA_STAGES;
            mbar_wait(&kv_full[s], (t / FA_STAGES) & 1);
            tc_fence_after();
            const uint32_t k_base = smem_u32(smem_k + s * FA_TILE_BYTES), v_base = smem_u32(smem_v + s * FA_TILE_BYTES);
            // S = Q Kt (contraction over d = HD / 8 k-steps of 8, four per 32-column box).  Issued after PV(t-1), so it
            // cannot overwrite P(t-1) before that MMA has consumed it (the tensor pipe executes in issue order).
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < HD / 8; ++j) {
                    const uint32_t off = (j / 4) * FA_BOX_BYTES + (j % 4) * 32;
                    umma_tf32(tmem_base, make_smem_desc(q_base + off, 16, 1024, 2), make_smem_desc(k_base + off, 16, 1024, 2),
                              idesc_s, j != 0);
                }
                umma_commit(s_full);
            }
            __syncwarp();
            // O_tile = P V (contraction over the 128 keys = 16 k-steps of 8 TMEM columns / 8 V rows)
            mbar_wait(p_full, t & 1);
            tc_fence_after();
            if (elect_one()) {
#pragma unroll
                for (int j = 0; j < FA_KT / 8; ++j)
                    umma_tf32_ts(tmem_base + FA_O_COL, tmem_base + j * 8, make_smem_desc(v_base + j * 1024, v_lbo, 512, 1), idesc_o, j != 0);
                umma_commit(&kv_empty[s]);
                umma_commit(o_full);
            }
            __syncwarp();
        }
    } else {
        const int q = warp & 3;
        const int row = q0 + q * 32 + lane;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16);
        float m = -CUDART_INF_F, l = 0.0f;
        float acc[HD];
#pragma unroll
        for (int i = 0; i < HD; ++i) acc[i] = 0.0f;
        for (int t = 0; t < ntiles; ++t) {
            const int valid = min(FA_KT, Lk - t * FA_KT);
            mbar_wait(s_full, t & 1);
            tc_fence_after();
            // pass 1: row maximum of the raw scores (next chunk's TMEM load in flight while this one is reduced)
            const bool full_tile = valid == FA_KT;            // only the last tile of a ragged Lk needs masking
            uint32_t ra[32], rb[32];
            float mx = -CUDART_INF_F;
            tmem_ld32_issue(lane_addr, ra);
#pragma unroll
            for (int c = 0; c < FA_KT / 32; ++c) {
                uint32_t *cur = (c & 1) ? rb : ra, *nxt = (c & 1) ? ra : rb;
                tmem_ld32_wait(cur);
                if (c + 1 < FA_KT / 32) tmem_ld32_issue(lane_addr + (c + 1) * 32, nxt);
                if (full_tile) {
                    mx = fmaxf(mx, max32_tree(cur));              // 3-input max tree (depth 4) instead of a 32-deep chain
                } else {
#pragma unroll
                    for (int i = 0; i < 32; ++i) mx = fmaxf(mx, (c * 32 + i < valid) ? __uint_as_float(cur[i]) : -CUDART_INF_F);
                }
            }
            const float m_new = fmaxf(m, mx * scale_log2);
            const float alpha = ex2_approx(m - m_new);            // first tile: exp2(-inf) = 0
            // pass 2: P = exp2(s*c - m_new) rounded to tf32, written back over S
            float psum = 0.0f;
            tmem_ld32_issue(lane_addr, ra);
#pragma unroll
            for (int c = 0; c < FA_KT / 32; ++c) {
                uint32_t *cur = (c & 1) ? rb : ra, *nxt = (c & 1) ? ra : rb;
                tmem_ld32_wait(cur);
                if (c + 1 < FA_KT / 32) tmem_ld32_issue(lane_addr + (c + 1) * 32, nxt);
                // keep the 10 mantissa bits the tf32 MMA will read (one LOP on the ALU pipe; cvt.rna would compete with
                // ex2 for the XU pipe) and sum exactly those weights, so numerator and denominator of the softmax use
                // identical values and the truncation bias cancels.  Packed FFMA2 / FADD2 and four independent partial
                // sums keep the dependency chains short.
                if (!full_tile) {
#pragma unroll
                    for (int i = 0; i < 32; ++i) if (c * 32 + i >= valid) cur[i] = 0xFF800000u;          // -inf -> exp2 = 0
                }
                const uint64_t sc2 = pack_f32x2(scale_log2, scale_log2), nm2 = pack_f32x2(-m_new, -m_new);
                uint64_t ps_a = pack_f32x2(0.0f, 0.0f), ps_b = ps_a;
#pragma unroll
                for (int i = 0; i < 32; i += 4) {
                    float x0, x1, x2, x3;
                    unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1])), sc2, nm2), x0, x1);
                    unpack_f32x2(fma_f32x2(pack_f32x2(__uint_as_float(cur[i + 2]), __uint_as_float(cur[i + 3])), sc2, nm2), x2, x3);
                    cur[i] = __float_as_uint(ex2_approx(x0)) & 0xFFFFE000u;
                    cur[i + 1] = __float_as_uint(ex2_approx(x1)) & 0xFFFFE000u;
                    cur[i + 2] = __float_as_uint(ex2_approx(x2)) & 0xFFFFE000u;
                    cur[i + 3] = __float_as_uint(ex2_approx(x3)) & 0xFFFFE000u;
                    ps_a = add_f32x2(ps_a, pack_f32x2(__uint_as_float(cur[i]), __uint_as_float(cur[i + 1])));
                    ps_b = add_f32x2(ps_b, pack_f32x2(__uint_as_float(cur[i + 2]), __uint_as_float(cur[i + 3])));
                }
                {
                    float s0, s1;
                    unpack_f32x2(add_f32x2(ps_a, ps_b), s0, s1);
                    psum += s0 + s1;
                }
                tmem_st32_u(lane_addr + c * 32, cur);
            }
            tmem_st_wait();
            tc_fence_before();
            mbar_arrive(p_full);
            l = fmaf(l, alpha, psum);
            m = m_new;
            // O_tile
            mbar_wait(o_full, t & 1);
            tc_fence_after();
#pragma unroll
            for (int c = 0; c < NB; ++c) {                    // 32 columns at a time: one x32 load's registers live
                float ot[32];
                tmem_ld32(lane_addr + FA_O_COL + c * 32, ot);
#pragma unroll
                for (int i = 0; i < 32; ++i) acc[c * 32 + i] = fmaf(acc[c * 32 + i], alpha, ot[i]);
            }
        }
        if (row < Lq) {
            const float inv = 1.0f / l;
            float *dst = o + (((size_t)b * H + h) * Lq + row) * HD;
#pragma unroll
            for (int i = 0; i < HD; i += 4) {
                float4 w = make_float4(acc[i] * inv, acc[i + 1] * inv, acc[i + 2] * inv, acc[i + 3] * inv);
                if (round_out) { w.x = tf32_rn(w.x); w.y = tf32_rn(w.y); w.z = tf32_rn(w.z); w.w = tf32_rn(w.w); }
                *reinterpret_cast<float4 *>(dst + i) = w;
            }
            lse[((size_t)b * H + h) * Lq + row] = m + log2f(l);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, FA_TMEM_COLS);
}

bool attention_umma_eligible(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp)
{
    auto al = [](const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; };
    return (d == 32 || d == 64) && al(qp) && al(kp) && al(vp) && B >= 1 && Lq >= 1 && Lk >= 1 && H >= 1;      // (TMA boxes may exceed the tensor: out-of-range rows are zero-filled)
}

namespace {

template <int HD>
int launch_fwd_umma(int B, int H, int Lq, int Lk, const float *qp, const float *kp, const float *vp, float *o, float *lse,
                    int round_out, cudaStream_t s)
{
    const int D = H * HD;
    CUtensorMap mq, mk, mv;
    bool ok = encode_tensor_map_2d(&mq, qp, (long long)B * Lq, D, D, 32, FA_BM, false);
    ok = ok && encode_tensor_map_2d(&mk, kp, (long long)B * Lk, D, D, 32, FA_KT, false);
    ok = ok && encode_tensor_map_2d(&mv, vp, (long long)B * Lk, D, D, 32, FA_KT, true);
    BDETR_REQUIRE(ok, BDETR_E_CUDA, "cuTensorMapEncodeTiled failed");
    const size_t smem = (size_t)(1 + 2 * FA_STAGES) * (FA_KT * HD * 4) + 16 * 8 + 16 + 1024;
    static bool optin = false;
    if (!optin) {
        BDETR_CUDA(cudaFuncSetAttribute(attention_fwd_umma_kernel<HD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        optin = true;
    }
    const float scale_log2 = (1.0f / sqrtf((float)HD)) * 1.4426950408889634f;
    dim3 grid(ceil_div(Lq, FA_BM), H, B);
    launch_k(attention_fwd_umma_kernel<HD>, grid, FA_THREADS, smem, s, mq, mk, mv, H, Lq, Lk, o, lse, scale_log2, round_out);
    BDETR_CHECK_LAUNCH("attention_fwd_umma_kernel");
    return BDETR_OK;
}

}  // namespace

int launch_attention_fwd_umma(int B, int H, int Lq, int Lk, int d, const float *qp, const float *kp, const float *vp,
                              float *o, float *lse, int round_out, cudaStream_t s)
{
    BDETR_REQUIRE(d == 32 || d == 64, BDETR_E_UNSUPPORTED, "head dim must be 32 or 64 (D/H)");
    return d == 64 ? launch_fwd_umma<64>(B, H, Lq, Lk, qp, kp, vp, o, lse, round_out, s)
                   : launch_fwd_umma<32>(B, H, Lq, Lk, qp, kp, vp, o, lse, round_out, s);
}

}  // namespace bdetr
