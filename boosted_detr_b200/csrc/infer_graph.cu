// Graph-captured inference with the early exit decided on the device (conditional graph nodes, CUDA 12.4+).
//
// The eager early exit (BoostedDETR._early_exit) copies the per-image confidences to the host after every boosted block
// and synchronises before it issues the next block.  Here the same decision is a kernel: it reads the confidences that
// bdetr_inverse_tokenize wrote for boundary i and sets the condition of the IF node that gates block i + 1.  The host
// captures the forward as segments (S0 = prologue + block 0, Sk = block k + its decide launch, E = the output select)
// and bdetr_exit_graph_build stitches them into
//     child(S0) -> IF(h1){child(S1)} -> IF(h2){child(S2)} -> ... -> child(E)
// Every handle resets to 0 at launch (cudaGraphCondAssignDefault), so a block that does not run leaves every later IF
// at 0 as well: the blocks after the exit are skipped as a whole.
#include <vector>
#include "kernels.cuh"

//
// Per-image early exit (bdetr_image_exit_*): after boundary i the images that are still running are gathered to the
// front of the batch and block i + 1 runs at that smaller batch.  The plan kernel decides which slots leave and the new
// order; the compaction kernel writes the leaving images' running predictions to the outputs at their original index and
// gathers the survivors' encoder output and running predictions into the next block's input buffers.  In a graph the
// plan sets the value of a SWITCH node whose bodies are the next block captured at every batch size
// (bdetr_switch_graph_*).
struct bdetr_exit_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<cudaGraphConditionalHandle> handles;
    int branches = 0;                    // 0: IF chain (bdetr_exit_graph_create); > 0: SWITCH chain of that many bodies each
};

namespace bdetr {

// Decision after boosted block `boundary` (one CTA).  The exit rule is the eager one bit for bit: exit when at least
// min_blocks blocks have run, a threshold is set and EVERY image has image_conf >= threshold (float32 compare; a NaN
// confidence is not confident).  exit_block = boundary on exit, n_blocks - 1 otherwise (a later boundary overwrites it).
__global__ void __launch_bounds__(128)
early_exit_decide_kernel(int B, int boundary, int n_blocks, const float *__restrict__ image_conf, const float *__restrict__ threshold,
                         const int32_t *__restrict__ min_blocks, const int32_t *__restrict__ threshold_set,
                         cudaGraphConditionalHandle next_block, int32_t *__restrict__ exit_block, float *__restrict__ conf_out)
{
    pdl_sync();
    const float thr = *threshold;
    int confident = 1;
    for (int b = threadIdx.x; b < B; b += blockDim.x) {
        const float c = image_conf[b];
        conf_out[b] = c;
        confident &= (c >= thr) ? 1 : 0;
    }
    const int all_confident = __syncthreads_and(confident);
    if (threadIdx.x == 0) {
        const bool go_on = boundary + 1 < *min_blocks || *threshold_set == 0 || !all_confident;
        *exit_block = go_on ? n_blocks - 1 : boundary;
        if (next_block) cudaGraphSetConditional(next_block, go_on ? 1u : 0u);
    }
}

struct ExitSources {
    const float *p[3 * BDETR_MAX_EXIT_BLOCKS];
};

// out_k = running prediction k of block *exit_block, for k = category, attribute, box
__global__ void __launch_bounds__(256)
select_exit_predictions_kernel(int n_blocks, long long n_cat, long long n_attr, long long n_box, ExitSources src,
                               const int32_t *__restrict__ exit_block, float *__restrict__ cat, float *__restrict__ attr,
                               float *__restrict__ box)
{
    pdl_sync();
    int e = *exit_block;
    e = e < 0 ? 0 : (e >= n_blocks ? n_blocks - 1 : e);
    const float *sc = src.p[3 * e], *sa = src.p[3 * e + 1], *sb = src.p[3 * e + 2];
    const long long total = n_cat + n_attr + n_box;
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < total; j += (long long)gridDim.x * blockDim.x) {
        if (j < n_cat) cat[j] = sc[j];
        else if (j < n_cat + n_attr) attr[j - n_cat] = sa[j - n_cat];
        else box[j - n_cat - n_attr] = sb[j - n_cat - n_attr];
    }
}

// The per-image exit state (int32 words; layout in include/bdetr.h, bdetr_image_exit_state_bytes).
struct ImageExitState {
    int32_t *n_active, *counts, *exit_block, *order, *src, *flag;
    float *conf;
    __host__ __device__ ImageExitState(int32_t *st, int B, int n_blocks)
    {
        n_active = st;
        counts = st + 1;
        exit_block = counts + n_blocks;
        conf = reinterpret_cast<float *>(exit_block + B);
        order = reinterpret_cast<int32_t *>(conf + B);
        src = order + 2 * B;
        flag = src + B;
    }
};
enum : int32_t { SLOT_RIDER = 0, SLOT_STAYS = 1, SLOT_EXITS = 2 };

// Plan of boundary `boundary` (one CTA).  Slot s of the k_in running slots holds image order_in[s] (a rider, an image that
// has already left and only fills the batch up to k_min, is stored as ~image); boundary 0 starts from the identity.  A live
// image leaves under the eager rule applied to it alone: a threshold is set, boundary + 1 >= min_blocks, and its float32
// confidence >= the float32 threshold (a NaN is not confident).  The survivors keep their relative order, and when fewer
// than k_min survive, the first non-surviving slots ride along.
__global__ void __launch_bounds__(256)
image_exit_plan_kernel(int B, int n_blocks, int k_min, int boundary, int k_in, const float *__restrict__ image_conf,
                       const float *__restrict__ threshold, const int32_t *__restrict__ min_blocks,
                       const int32_t *__restrict__ threshold_set, cudaGraphConditionalHandle next_switch, int32_t *state)
{
    pdl_sync();
    ImageExitState st(state, B, n_blocks);
    const int32_t *order_in = boundary == 0 ? nullptr : st.order + ((boundary - 1) & 1) * B;
    int32_t *order_out = st.order + (boundary & 1) * B;
    const float thr = *threshold;
    const bool checked = *threshold_set != 0 && boundary + 1 >= *min_blocks;
    if (order_in == nullptr) {                      // first boundary of the call: every image runs to the last block so far
        for (int b = threadIdx.x; b < B; b += blockDim.x) {
            st.exit_block[b] = n_blocks - 1;
            st.conf[b] = __int_as_float(0x7fc00000);
        }
    }
    __syncthreads();
    for (int s = threadIdx.x; s < k_in; s += blockDim.x) {
        const int e = order_in ? order_in[s] : s;
        int32_t f = SLOT_RIDER;
        if (e >= 0) {
            f = SLOT_STAYS;
            if (checked) {
                const float c = image_conf[s];
                st.conf[e] = c;
                if (c >= thr) {
                    f = SLOT_EXITS;
                    st.exit_block[e] = boundary;
                }
            }
        }
        st.flag[s] = f;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int n_stay = 0;
        for (int s = 0; s < k_in; ++s) n_stay += st.flag[s] == SLOT_STAYS;
        const int k_out = n_stay == 0 ? 0 : max(n_stay, min(k_min, k_in));
        int j = 0;
        for (int s = 0; s < k_in; ++s)
            if (st.flag[s] == SLOT_STAYS) {
                order_out[j] = order_in ? order_in[s] : s;
                st.src[j++] = s;
            }
        for (int s = 0; s < k_in && j < k_out; ++s)
            if (st.flag[s] != SLOT_STAYS) {
                const int e = order_in ? order_in[s] : s;
                order_out[j] = e >= 0 ? ~e : e;
                st.src[j++] = s;
            }
        *st.n_active = k_out;
        st.counts[boundary] = k_in;
        st.counts[boundary + 1] = k_out;
        if (k_out == 0)
            for (int b = boundary + 2; b < n_blocks; ++b) st.counts[b] = 0;
        if (next_switch) cudaGraphSetConditional(next_switch, k_out == 0 ? (unsigned)(B - k_min + 1) : (unsigned)(k_out - k_min));
    }
}

struct ExitRows {
    const float *in[4];        // x, category, attribute, box of the k_in running slots
    float *gathered[4];        // the same, gathered for the next block
    float *out[3];             // category, attribute, box outputs [B, Q, .] in the caller's image order
    long long len[4];          // floats per image of each
};

__device__ __forceinline__ void copy_row(float *__restrict__ dst, const float *__restrict__ src, long long n, long long t0, long long stride)
{
    if ((n & 3) == 0) {
        const float4 *s4 = reinterpret_cast<const float4 *>(src);
        float4 *d4 = reinterpret_cast<float4 *>(dst);
        for (long long j = t0; j < n / 4; j += stride) d4[j] = __ldg(s4 + j);
    } else {
        for (long long j = t0; j < n; j += stride) dst[j] = __ldg(src + j);
    }
}

// grid (gx, k_in, 2).  z = 0: new slot y <- old slot src[y] for y < n_active (x and the three running predictions);
// z = 1: slot y's running predictions -> the outputs when its image leaves here (after the last block: every live slot).
__global__ void __launch_bounds__(256)
image_exit_compact_kernel(int B, int n_blocks, int boundary, ExitRows r, const int32_t *state)
{
    pdl_sync();
    ImageExitState st(const_cast<int32_t *>(state), B, n_blocks);
    const bool last = boundary == n_blocks - 1;
    const int y = blockIdx.y;
    const long long t0 = (long long)blockIdx.x * blockDim.x + threadIdx.x, stride = (long long)gridDim.x * blockDim.x;
    if (blockIdx.z == 0) {
        if (last || y >= *st.n_active) return;
        const int s = st.src[y];
        for (int t = 0; t < 4; ++t) copy_row(r.gathered[t] + y * r.len[t], r.in[t] + s * r.len[t], r.len[t], t0, stride);
    } else {
        const int e = boundary == 0 ? y : st.order[((boundary - 1) & 1) * B + y];
        if (e < 0 || !(last || st.flag[y] == SLOT_EXITS)) return;
        for (int t = 1; t < 4; ++t) copy_row(r.out[t - 1] + e * r.len[t], r.in[t] + y * r.len[t], r.len[t], t0, stride);
    }
}

}  // namespace bdetr

using namespace bdetr;

#define BDETR_API extern "C" __attribute__((visibility("default")))

BDETR_API int bdetr_early_exit_decide(int B, int boundary, int n_blocks, const float *image_conf, const float *threshold,
                                      const int32_t *min_blocks, const int32_t *threshold_set, unsigned long long next_block,
                                      int32_t *exit_block, float *conf_out, void *stream)
{
    BDETR_REQUIRE(B > 0 && boundary >= 0 && boundary + 1 < n_blocks, BDETR_E_BAD_SHAPE, "need B > 0 and 0 <= boundary < n_blocks - 1");
    BDETR_REQUIRE(image_conf && threshold && min_blocks && threshold_set && exit_block && conf_out, BDETR_E_NULL, "null pointer");
    launch_k(early_exit_decide_kernel, 1, 128, 0, as_stream(stream), B, boundary, n_blocks, image_conf, threshold, min_blocks,
             threshold_set, (cudaGraphConditionalHandle)next_block, exit_block, conf_out);
    BDETR_CHECK_LAUNCH("early_exit_decide_kernel");
    return BDETR_OK;
}

BDETR_API int bdetr_select_exit_predictions(int n_blocks, int B, int Q, int C, int A, const float *const *cums,
                                            const int32_t *exit_block, float *cat, float *attr, float *box, void *stream)
{
    BDETR_REQUIRE(n_blocks >= 1 && n_blocks <= BDETR_MAX_EXIT_BLOCKS, BDETR_E_UNSUPPORTED, "n_blocks must be 1 .. BDETR_MAX_EXIT_BLOCKS");
    BDETR_REQUIRE(B > 0 && Q > 0 && C > 0 && A > 0, BDETR_E_BAD_SHAPE, "bad shape");
    BDETR_REQUIRE(cums && exit_block && cat && attr && box, BDETR_E_NULL, "null pointer");
    ExitSources src = {};
    for (int k = 0; k < 3 * n_blocks; ++k) {
        BDETR_REQUIRE(cums[k], BDETR_E_NULL, "null running-prediction pointer");
        src.p[k] = cums[k];
    }
    const long long M = (long long)B * Q, total = M * (C + A + 4);
    const int grid = (int)((total + 255) / 256 < 1184 ? (total + 255) / 256 : 1184);
    launch_k(select_exit_predictions_kernel, grid, 256, 0, as_stream(stream), n_blocks, M * C, M * A, M * 4, src, exit_block,
             cat, attr, box);
    BDETR_CHECK_LAUNCH("select_exit_predictions_kernel");
    return BDETR_OK;
}

BDETR_API size_t bdetr_image_exit_state_bytes(int B, int n_blocks)
{
    if (B <= 0 || n_blocks < 2) return 0;
    return sizeof(int32_t) * (1 + (size_t)n_blocks + 6 * (size_t)B);
}

BDETR_API int bdetr_image_exit_plan(int B, int n_blocks, int k_min, int boundary, int k_in, const float *image_conf,
                                    const float *threshold, const int32_t *min_blocks, const int32_t *threshold_set,
                                    unsigned long long next_switch, int32_t *state, void *stream)
{
    BDETR_REQUIRE(B > 0 && boundary >= 0 && boundary + 1 < n_blocks, BDETR_E_BAD_SHAPE, "need B > 0 and 0 <= boundary < n_blocks - 1");
    BDETR_REQUIRE(k_min >= 1 && k_min <= k_in && k_in <= B && (boundary > 0 || k_in == B), BDETR_E_BAD_SHAPE,
                  "need 1 <= k_min <= k_in <= B, and k_in == B at boundary 0");
    BDETR_REQUIRE(image_conf && threshold && min_blocks && threshold_set && state, BDETR_E_NULL, "null pointer");
    launch_k(image_exit_plan_kernel, 1, 256, 0, as_stream(stream), B, n_blocks, k_min, boundary, k_in, image_conf, threshold,
             min_blocks, threshold_set, (cudaGraphConditionalHandle)next_switch, state);
    BDETR_CHECK_LAUNCH("image_exit_plan_kernel");
    return BDETR_OK;
}

BDETR_API int bdetr_image_exit_compact(int B, int n_blocks, int boundary, int k_in, int Q, int C, int A, long long x_row,
                                       const float *x_in, const float *const *cum_in, float *x_out, float *const *cum_out,
                                       float *const *out, const int32_t *state, void *stream)
{
    BDETR_REQUIRE(B > 0 && n_blocks >= 2 && boundary >= 0 && boundary < n_blocks && k_in >= 1 && k_in <= B, BDETR_E_BAD_SHAPE,
                  "need 0 <= boundary < n_blocks, n_blocks >= 2 and 1 <= k_in <= B");
    BDETR_REQUIRE(Q > 0 && C > 0 && A > 0 && x_row > 0, BDETR_E_BAD_SHAPE, "bad shape");
    const bool last = boundary == n_blocks - 1;
    BDETR_REQUIRE(cum_in && out && state && (last || (x_in && x_out && cum_out)), BDETR_E_NULL, "null pointer");
    ExitRows r = {};
    r.in[0] = x_in;
    r.gathered[0] = x_out;
    r.len[0] = x_row;
    const long long lens[3] = {(long long)Q * C, (long long)Q * A, (long long)Q * 4};
    for (int t = 0; t < 3; ++t) {
        BDETR_REQUIRE(cum_in[t] && out[t] && (last || cum_out[t]), BDETR_E_NULL, "null pointer");
        r.in[t + 1] = cum_in[t];
        r.gathered[t + 1] = last ? nullptr : cum_out[t];
        r.out[t] = out[t];
        r.len[t + 1] = lens[t];
    }
    const long long longest = last ? lens[0] : (x_row > lens[0] ? x_row : lens[0]);
    long long gx = (longest / 4 + 255) / 256;
    const long long cap = 1184 / k_in > 1 ? 1184 / k_in : 1;
    gx = gx < 1 ? 1 : (gx > cap ? cap : gx);
    launch_k(image_exit_compact_kernel, dim3((unsigned)gx, (unsigned)k_in, 2), 256, 0, as_stream(stream), B, n_blocks, boundary, r,
             state);
    BDETR_CHECK_LAUNCH("image_exit_compact_kernel");
    return BDETR_OK;
}

static int exit_graph_create(int n_boundaries, int branches, bdetr_exit_graph **out, unsigned long long *handles)
{
    *out = nullptr;
    bdetr_exit_graph *g = new bdetr_exit_graph;
    g->branches = branches;
    cudaError_t e = cudaGraphCreate(&g->graph, 0);
    for (int i = 0; e == cudaSuccess && i < n_boundaries; ++i) {
        cudaGraphConditionalHandle h = 0;
        // default = branches: a SWITCH whose plan never ran matches no body (an IF handle defaults to 0: not taken)
        e = cudaGraphConditionalHandleCreate(&h, g->graph, (unsigned)branches, cudaGraphCondAssignDefault);
        g->handles.push_back(h);
        handles[i] = (unsigned long long)h;
    }
    if (e != cudaSuccess) {
        set_error("bdetr_exit_graph_create: %s", cudaGetErrorString(e));
        if (g->graph) cudaGraphDestroy(g->graph);
        delete g;
        return BDETR_E_CUDA;
    }
    *out = g;
    return BDETR_OK;
}

BDETR_API int bdetr_exit_graph_create(int n_boundaries, bdetr_exit_graph **out, unsigned long long *handles)
{
    BDETR_REQUIRE(out && (handles || n_boundaries == 0), BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(n_boundaries >= 0 && n_boundaries < BDETR_MAX_EXIT_BLOCKS, BDETR_E_UNSUPPORTED,
                  "n_boundaries must be 0 .. BDETR_MAX_EXIT_BLOCKS - 1");
    return exit_graph_create(n_boundaries, 0, out, handles);
}

BDETR_API int bdetr_switch_graph_create(int n_boundaries, int n_branches, bdetr_exit_graph **out, unsigned long long *handles)
{
    BDETR_REQUIRE(out && handles, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(n_boundaries >= 1 && n_boundaries < BDETR_MAX_EXIT_BLOCKS && n_branches >= 1, BDETR_E_UNSUPPORTED,
                  "n_boundaries must be 1 .. BDETR_MAX_EXIT_BLOCKS - 1 and n_branches >= 1");
    int driver = 0;
    BDETR_CUDA(cudaDriverGetVersion(&driver));
    BDETR_REQUIRE(driver >= 12080, BDETR_E_UNSUPPORTED, "SWITCH graph nodes need a CUDA 12.8 driver or newer");
    return exit_graph_create(n_boundaries, n_branches, out, handles);
}

BDETR_API int bdetr_switch_graph_build(bdetr_exit_graph *g, void *const *segments, int n_segments)
{
    BDETR_REQUIRE(g && segments, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(!g->exec, BDETR_E_UNSUPPORTED, "the graph is already built");
    BDETR_REQUIRE(g->branches > 0, BDETR_E_UNSUPPORTED, "created by bdetr_exit_graph_create: build it with bdetr_exit_graph_build");
    const int nb = (int)g->handles.size(), nbr = g->branches;
    BDETR_REQUIRE(n_segments == 1 + nb * nbr, BDETR_E_BAD_SHAPE, "need 1 + n_boundaries * n_branches segments");
    for (int k = 0; k < n_segments; ++k) BDETR_REQUIRE(segments[k], BDETR_E_NULL, "null segment graph");
    cudaGraphNode_t prev = nullptr, node = nullptr;
    BDETR_CUDA(cudaGraphAddChildGraphNode(&node, g->graph, nullptr, 0, (cudaGraph_t)segments[0]));
    prev = node;
    for (int i = 0; i < nb; ++i) {
        cudaGraphNodeParams p = {};
        p.type = cudaGraphNodeTypeConditional;
        p.conditional.handle = g->handles[i];
        p.conditional.type = cudaGraphCondTypeSwitch;
        p.conditional.size = (unsigned)nbr;
        BDETR_CUDA(cudaGraphAddNode(&node, g->graph, &prev, 1, &p));
        for (int v = 0; v < nbr; ++v) {
            cudaGraphNode_t child = nullptr;
            BDETR_CUDA(cudaGraphAddChildGraphNode(&child, p.conditional.phGraph_out[v], nullptr, 0, (cudaGraph_t)segments[1 + i * nbr + v]));
        }
        prev = node;
    }
    cudaGraphInstantiateParams ip = {};
    const cudaError_t e = cudaGraphInstantiateWithParams(&g->exec, g->graph, &ip);
    if (e != cudaSuccess) {
        g->exec = nullptr;
        set_error("bdetr_switch_graph_build: instantiation failed: %s (instantiate result %d)", cudaGetErrorString(e), (int)ip.result_out);
        return BDETR_E_CUDA;
    }
    return BDETR_OK;
}

BDETR_API int bdetr_exit_graph_build(bdetr_exit_graph *g, void *const *segments, int n_segments)
{
    BDETR_REQUIRE(g && segments, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(!g->exec, BDETR_E_UNSUPPORTED, "the graph is already built");
    BDETR_REQUIRE(g->branches == 0, BDETR_E_UNSUPPORTED, "created by bdetr_switch_graph_create: build it with bdetr_switch_graph_build");
    const int nb = (int)g->handles.size();
    BDETR_REQUIRE(n_segments == nb + 2, BDETR_E_BAD_SHAPE, "need n_boundaries + 2 segments (S0, S1 .. S_n, E)");
    for (int k = 0; k < n_segments; ++k) BDETR_REQUIRE(segments[k], BDETR_E_NULL, "null segment graph");
    cudaGraphNode_t prev = nullptr, node = nullptr;
    BDETR_CUDA(cudaGraphAddChildGraphNode(&node, g->graph, nullptr, 0, (cudaGraph_t)segments[0]));
    prev = node;
    for (int k = 1; k <= nb; ++k) {
        cudaGraphNodeParams p = {};
        p.type = cudaGraphNodeTypeConditional;
        p.conditional.handle = g->handles[k - 1];
        p.conditional.type = cudaGraphCondTypeIf;
        p.conditional.size = 1;
        BDETR_CUDA(cudaGraphAddNode(&node, g->graph, &prev, 1, &p));
        cudaGraphNode_t child = nullptr;
        BDETR_CUDA(cudaGraphAddChildGraphNode(&child, p.conditional.phGraph_out[0], nullptr, 0, (cudaGraph_t)segments[k]));
        prev = node;
    }
    BDETR_CUDA(cudaGraphAddChildGraphNode(&node, g->graph, &prev, 1, (cudaGraph_t)segments[n_segments - 1]));
    cudaGraphInstantiateParams ip = {};
    const cudaError_t e = cudaGraphInstantiateWithParams(&g->exec, g->graph, &ip);
    if (e != cudaSuccess) {
        g->exec = nullptr;
        set_error("bdetr_exit_graph_build: instantiation failed: %s (instantiate result %d)", cudaGetErrorString(e), (int)ip.result_out);
        return BDETR_E_CUDA;
    }
    return BDETR_OK;
}

BDETR_API int bdetr_exit_graph_launch(bdetr_exit_graph *g, void *stream)
{
    BDETR_REQUIRE(g, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(g->exec, BDETR_E_UNSUPPORTED, "bdetr_exit_graph_build has not succeeded");
    BDETR_CUDA(cudaGraphLaunch(g->exec, as_stream(stream)));
    return BDETR_OK;
}

BDETR_API int bdetr_exit_graph_destroy(bdetr_exit_graph *g)
{
    if (!g) return BDETR_OK;
    cudaError_t e = cudaSuccess;
    if (g->exec) e = cudaGraphExecDestroy(g->exec);
    const cudaError_t e2 = cudaGraphDestroy(g->graph);
    delete g;
    BDETR_CUDA(e);
    BDETR_CUDA(e2);
    return BDETR_OK;
}
