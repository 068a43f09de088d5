// Host-side launchers for the MLP layer kernels (mlp.cuh), the flat parameter layout and the
// forward-only entry point.
#include "umma.cuh"
#include "internal.h"
#include <stdlib.h>

namespace ppoaf {

static inline bool vec4_ok(const float* p, int ld, int contig_extent) {
    return (reinterpret_cast<uintptr_t>(p) % 16 == 0) && (ld % 4 == 0) && (contig_extent % 4 == 0);
}

// Called from ppoaf_runtime_init (so that the attribute calls normally happen before any stream capture) and, for
// callers of the C ABI that never initialise the runtime, lazily by the first launch.
static bool g_gemm_configured = false;
void configure_gemm_kernels() {
    g_gemm_configured = true;
    cudaFuncSetAttribute(grouped_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kGemmSmemBytes));
    cudaFuncSetAttribute(umma::umma_grouped_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         int(umma::kUmmaSmemBytes));
}

static inline int tile_m(int backend) { return backend == GEMM_BACKEND_TCGEN05 ? umma::kUM : kBM; }
static inline int tile_n(int backend) { return backend == GEMM_BACKEND_TCGEN05 ? umma::kUN : kBN; }

GemmGroup::GemmGroup(int backend_) : args(new GroupedGemmArgs()), n_tiles(0), backend(backend_) { args->n_problems = 0; }
GemmGroup::~GemmGroup() { delete args; }
static_assert(kMaxGroupHost == kMaxGroup, "internal.h and mlp.cuh disagree on the group size");

static GemmProblem* next_problem(GemmGroup* grp, int M, int N) {
    GemmProblem* g = &grp->args->p[grp->args->n_problems++];
    memset(g, 0, sizeof(*g));
    g->tiles_n = (N + tile_n(grp->backend) - 1) / tile_n(grp->backend);
    g->tile_begin = grp->n_tiles;
    grp->n_tiles += g->tiles_n * ((M + tile_m(grp->backend) - 1) / tile_m(grp->backend));
    return g;
}

void GemmGroup::add_forward(const float* X, int ldx, const int64_t* idx, const float* W, const float* b, float* Y,
                            int rows, int in, int out, int act, bool w_static) {
    GemmProblem* g = next_problem(this, rows, out);
    g->b_static = w_static ? 1 : 0;
    g->A = X; g->lda = ldx; g->B = W; g->ldb = in; g->C = Y; g->ldc = out;
    g->M = rows; g->N = out; g->K = in;
    g->idxA = idx; g->bias = b; g->act = act;
    g->flavour = EPI_FWD * 4 + (vec4_ok(X, ldx, in) ? 2 : 0) + (vec4_ok(W, in, in) ? 1 : 0);
}

void GemmGroup::add_backward_x(const float* dZ, const float* W, const float* Xact, float* dX, int rows, int in,
                               int out, int act) {
    GemmProblem* g = next_problem(this, rows, in);
    g->A = dZ; g->lda = out; g->B = W; g->ldb = in; g->C = dX; g->ldc = in;
    g->M = rows; g->N = in; g->K = out;
    g->aux = Xact; g->ldaux = in; g->act = act;
    g->b_static = 1;                      // W is only written by the optimizer, several launches back
    g->flavour = EPI_BWD_X * 4 + (vec4_ok(dZ, out, out) ? 2 : 0) + (vec4_ok(W, in, in) ? 1 : 0);
}

int backward_w_tiles(int in, int out) {
    return ((in + kBN - 1) / kBN) * ((out + kBM - 1) / kBM);
}

int GemmGroup::add_backward_w(const float* dZ, const float* X, int ldx, const int64_t* idx, float* dW, float* db,
                              int rows, int in, int out, double* sq_out, bool x_static) {
    GemmProblem* g = next_problem(this, out, in);
    g->b_static = (x_static && idx == nullptr) ? 1 : 0;
    g->A = dZ; g->lda = out; g->B = X; g->ldb = ldx; g->C = dW; g->ldc = in;
    g->M = out; g->N = in; g->K = rows;
    g->idxB = idx; g->dbias = db; g->sq_out = sq_out;
    g->flavour = EPI_BWD_W * 4 + (vec4_ok(dZ, out, out) ? 2 : 0) + (vec4_ok(X, ldx, in) ? 1 : 0);
    return backward_w_tiles(in, out);
}

int GemmGroup::launch(const int32_t* cursor, int cursor_stride, cudaStream_t s, int n_mirror, const int64_t* mirror_delta) {
    if (n_tiles == 0) return 0;
    if (!g_gemm_configured) configure_gemm_kernels();
    args->cursor = cursor;
    args->cursor_stride = cursor_stride;
    args->mirror.n = n_mirror;
    for (int q = 0; q < n_mirror && q < PPOAF_MAX_MIRROR; ++q) args->mirror.delta[q] = mirror_delta[q];
    if (backend == GEMM_BACKEND_TCGEN05) {
        for (int i = 0; i < args->n_problems; ++i)
            PPOAF_CHECK_ARG(args->p[i].flavour >> 2 == EPI_FWD, "GemmGroup::launch: the tcgen05 tiles run forward problems only");
        launch_chain(umma::umma_grouped_gemm_kernel, dim3(n_tiles), dim3(umma::kUThreads + 32), umma::kUmmaSmemBytes, s, *args);
        PPOAF_CHECK_LAUNCH("umma_grouped_gemm_kernel");
    } else {
        launch_chain(grouped_gemm_kernel, dim3(n_tiles), dim3(kThreads), kGemmSmemBytes, s, *args);
        PPOAF_CHECK_LAUNCH("grouped_gemm_kernel");
    }
    return 0;
}

__global__ void softmax_rows_kernel(float* __restrict__ y, int rows, int n) {
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= rows) return;
    float* p = y + int64_t(r) * n;
    float mx = p[0];
    for (int j = 1; j < n; ++j) mx = fmaxf(mx, p[j]);
    float s = 0.f;
    for (int j = 0; j < n; ++j) { const float e = expf(p[j] - mx); p[j] = e; s += e; }
    for (int j = 0; j < n; ++j) p[j] = p[j] / s;
}

// Rows wider than 64 columns: one warp per row, the lanes striding over it (sums in a different order from
// softmax_rows_kernel, so results can differ from it in the last bits)
__global__ void __launch_bounds__(256) softmax_rows_wide_kernel(float* __restrict__ y, int rows, int n) {
    const int lane = threadIdx.x & 31, r = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= rows) return;
    float* p = y + int64_t(r) * n;
    float mx = -INFINITY;
    for (int j = lane; j < n; j += 32) mx = fmaxf(mx, p[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(kFull, mx, o));
    float s = 0.f;
    for (int j = lane; j < n; j += 32) { const float e = expf(p[j] - mx); p[j] = e; s += e; }
    s = warp_sum(s);
    for (int j = lane; j < n; j += 32) p[j] = p[j] / s;
}

// Backend of the forward-only launches (ppoaf_mlp_forward; the update always runs the FFMA tiles): FFMA tiles (default:
// faster up to 512 rows, DESIGN.md §3.3) or the tcgen05 3xTF32 tiles (PPOAF_GEMM=tcgen05 or ppoaf_set_gemm_backend(1)).
static int g_backend = -1;
int gemm_backend() {
    if (g_backend < 0) {
        const char* e = getenv("PPOAF_GEMM");
        g_backend = (e && (strcmp(e, "tcgen05") == 0 || strcmp(e, "umma") == 0)) ? GEMM_BACKEND_TCGEN05 : GEMM_BACKEND_FFMA;
    }
    return g_backend;
}

int64_t param_layout(const ppoaf_mlp_desc* net, int32_t log_std_dim, int64_t* offsets) {
    int64_t off = 0;
    for (int l = 0; l < net->n_layers; ++l) {
        const int64_t w = int64_t(net->dims[l]) * net->dims[l + 1];
        if (offsets) offsets[2 * l] = off;
        off += (w + 3) / 4 * 4;
        if (offsets) offsets[2 * l + 1] = off;
        off += (int64_t(net->dims[l + 1]) + 3) / 4 * 4;
    }
    if (offsets) offsets[2 * net->n_layers] = off;
    if (log_std_dim > 0) off += (int64_t(log_std_dim) + 3) / 4 * 4;
    return off;
}

int check_mlp_desc(const ppoaf_mlp_desc* net, const char* who) {
    PPOAF_CHECK_ARG(net != nullptr, "%s: null mlp desc", who);
    PPOAF_CHECK_ARG(net->n_layers >= 1 && net->n_layers <= PPOAF_MAX_LAYERS, "%s: n_layers out of range", who);
    for (int l = 0; l <= net->n_layers; ++l) PPOAF_CHECK_ARG(net->dims[l] > 0, "%s: dims[%d] must be > 0", who, l);
    PPOAF_CHECK_ARG(net->activation >= PPOAF_ACT_IDENTITY && net->activation <= PPOAF_ACT_TANH,
                    "%s: unknown activation", who);
    return 0;
}

}  // namespace ppoaf

using namespace ppoaf;

extern "C" int64_t ppoaf_param_layout(const ppoaf_mlp_desc* net, int32_t log_std_dim, int64_t* offsets) {
    if (check_mlp_desc(net, "ppoaf_param_layout")) return -1;
    return param_layout(net, log_std_dim, offsets);
}

extern "C" size_t ppoaf_mlp_forward_workspace_bytes(const ppoaf_mlp_desc* net, int32_t n_rows) {
    if (!net || n_rows <= 0) return 64;
    int widest = 0;
    for (int l = 1; l <= net->n_layers; ++l) widest = net->dims[l] > widest ? net->dims[l] : widest;
    return 2 * align_up(size_t(n_rows) * widest * sizeof(float), 256) + 256;
}

extern "C" int ppoaf_mlp_forward(const ppoaf_mlp_desc* net, const float* params, const float* x, const int64_t* idx,
                                 int32_t n_rows, int softmax_out, float* y, void* workspace, size_t workspace_bytes,
                                 void* stream) {
    if (check_mlp_desc(net, "ppoaf_mlp_forward")) return 1;
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_mlp_forward: n_rows < 0");
    if (n_rows == 0) return 0;
    PPOAF_CHECK_ARG(workspace_bytes >= ppoaf_mlp_forward_workspace_bytes(net, n_rows),
                    "ppoaf_mlp_forward: workspace too small");
    PPOAF_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, "ppoaf_mlp_forward: workspace alignment");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t off[2 * PPOAF_MAX_LAYERS + 1];
    param_layout(net, 0, off);
    int widest = 0;
    for (int l = 1; l <= net->n_layers; ++l) widest = net->dims[l] > widest ? net->dims[l] : widest;
    const size_t half = align_up(size_t(n_rows) * widest * sizeof(float), 256);
    float* buf[2] = {reinterpret_cast<float*>(workspace),
                     reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + half)};
    const float* in = x;
    const int64_t* in_idx = idx;
    for (int l = 0; l < net->n_layers; ++l) {
        const bool last = l + 1 == net->n_layers;
        float* out = last ? y : buf[l & 1];
        GemmGroup grp(gemm_backend());
        grp.add_forward(in, net->dims[l], in_idx, params + off[2 * l], params + off[2 * l + 1], out, n_rows,
                        net->dims[l], net->dims[l + 1], last ? PPOAF_ACT_IDENTITY : net->activation, l > 0);
        if (grp.launch(nullptr, 0, s)) return 2;
        in = out;
        in_idx = nullptr;
    }
    if (softmax_out) {
        const int n = net->dims[net->n_layers];
        if (n > 64)
            softmax_rows_wide_kernel<<<(n_rows + 7) / 8, 256, 0, s>>>(y, n_rows, n);
        else
            softmax_rows_kernel<<<(n_rows + 127) / 128, 128, 0, s>>>(y, n_rows, n);
        PPOAF_CHECK_LAUNCH("ppoaf_mlp_forward(softmax)");
    }
    return 0;
}

#ifdef PPOAF_GEMM_TIMING
extern "C" int ppoaf_debug_gemm_stamps(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, ppoaf::g_gemm_stamps, sizeof(long long) * 16) == cudaSuccess ? 0 : 1;
}
#endif

extern "C" int ppoaf_set_gemm_backend(int backend) {
    PPOAF_CHECK_ARG(backend == GEMM_BACKEND_FFMA || backend == GEMM_BACKEND_TCGEN05, "ppoaf_set_gemm_backend: 0 = ffma, 1 = tcgen05");
    g_backend = backend;
    return 0;
}
extern "C" int ppoaf_get_gemm_backend(void) { return gemm_backend(); }
