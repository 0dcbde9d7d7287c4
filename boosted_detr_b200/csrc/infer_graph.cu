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

struct bdetr_exit_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    std::vector<cudaGraphConditionalHandle> handles;
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

BDETR_API int bdetr_exit_graph_create(int n_boundaries, bdetr_exit_graph **out, unsigned long long *handles)
{
    BDETR_REQUIRE(out && (handles || n_boundaries == 0), BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(n_boundaries >= 0 && n_boundaries < BDETR_MAX_EXIT_BLOCKS, BDETR_E_UNSUPPORTED,
                  "n_boundaries must be 0 .. BDETR_MAX_EXIT_BLOCKS - 1");
    *out = nullptr;
    bdetr_exit_graph *g = new bdetr_exit_graph;
    cudaError_t e = cudaGraphCreate(&g->graph, 0);
    for (int i = 0; e == cudaSuccess && i < n_boundaries; ++i) {
        cudaGraphConditionalHandle h = 0;
        e = cudaGraphConditionalHandleCreate(&h, g->graph, 0, cudaGraphCondAssignDefault);
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

BDETR_API int bdetr_exit_graph_build(bdetr_exit_graph *g, void *const *segments, int n_segments)
{
    BDETR_REQUIRE(g && segments, BDETR_E_NULL, "null pointer");
    BDETR_REQUIRE(!g->exec, BDETR_E_UNSUPPORTED, "the graph is already built");
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
