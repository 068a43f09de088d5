// One PPO minibatch as a fixed kernel sequence (reference ppo.py:2292-2468 -> policies/ppo_policy.py:
// 891-952, 1012-1055), plus the library-wide utilities (error string, device info).
//
//   grads:  forward layer l of actor AND critic (one grouped launch per hidden layer)
//           ->  fused loss kernel: the two head layers, loss forward/backward, the heads' dX
//           ->  dW/db and dX of layer l of both networks (one grouped launch per l, top layer first; the heads' dW
//               rides in the first of them)
//   apply:  clip + Adam (one launch).  R > 1: the caller runs the fused exchange + clip + Adam kernel of peer.cu
//           instead (or, on the NCCL fallback, all-reduces `grads` first: then a norm pass precedes Adam).
//
// 8 launches per minibatch on one stream (10 when the head layers cannot be fused: loss.cu, loss_head_fusable), chained
// with programmatic dependent launch (common.cuh).  Every kernel reads the minibatch cursor from device memory, so ONE
// captured graph serves every full minibatch.
#include <stdarg.h>

#include "internal.h"
#include <stdlib.h>

namespace ppoaf {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

bool pdl_enabled() {
    static int cached = -1;
    if (cached < 0) { const char* e = getenv("PPOAF_PDL"); cached = (e && e[0] == '0') ? 0 : 1; }
    return cached != 0;
}

int sm_count() {
    static int cached = 0;
    if (cached > 0) return cached;
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) {
        cached = n;
        return n;
    }
    (void)cudaGetLastError();
    return 148;  // B200; only used for sizing queries when no device is visible
}

// ---- workspace carving ------------------------------------------------------------------------------
struct NetScratch {
    float* act[PPOAF_MAX_LAYERS + 1];  // act[l] = output of layer l-1 (act[0] unused: the input is gathered)
    float* dz[PPOAF_MAX_LAYERS + 1];   // dz[l]  = gradient w.r.t. the pre-activation of layer l-1's output
    float* dact[PPOAF_MAX_LAYERS + 1]; // dact[l] = act'(z) of hidden layer l-1's output (act_stores_derivative ids), or null
};
struct StepScratch {
    NetScratch actor, critic;
    float* loss_partials;
    unsigned int* loss_ticket;
    void* optim_ws;
    double* sq_actor;   // per-tile sums of squares of the actor's gradient (+1 slot for log_std)
    double* sq_critic;
    int n_sq_actor, n_sq_critic;
    size_t total;
};

static int count_sq_slots(const ppoaf_mlp_desc* net) {
    int n = 0;
    for (int l = 0; l < net->n_layers; ++l) n += backward_w_tiles(net->dims[l], net->dims[l + 1]);
    return n;
}

static void carve(const ppoaf_update_cfg* cfg, int max_batch, char* base, StepScratch* out) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    // control blocks first, at offsets that do not depend on the batch: they hold self-resetting tickets
    // that must stay zero between launches, so no activation buffer may ever alias them
    out->loss_ticket = reinterpret_cast<unsigned int*>(take(256));
    out->optim_ws = take(optim_workspace_bytes());
    out->n_sq_actor = count_sq_slots(&cfg->actor) + 1;
    out->n_sq_critic = count_sq_slots(&cfg->critic);
    out->sq_actor = reinterpret_cast<double*>(take(size_t(out->n_sq_actor) * sizeof(double)));
    out->sq_critic = reinterpret_cast<double*>(take(size_t(out->n_sq_critic) * sizeof(double)));
    out->loss_partials = reinterpret_cast<float*>(take(loss_workspace_bytes(max_batch, cfg->act_dim)));
    const ppoaf_mlp_desc* nets[2] = {&cfg->actor, &cfg->critic};
    NetScratch* ns[2] = {&out->actor, &out->critic};
    for (int k = 0; k < 2; ++k) {
        for (int l = 1; l <= nets[k]->n_layers; ++l) {
            const size_t rows = (l == nets[k]->n_layers && k == 1) ? size_t(2) * max_batch : size_t(max_batch);
            ns[k]->act[l] = reinterpret_cast<float*>(take(size_t(max_batch) * nets[k]->dims[l] * sizeof(float)));
            ns[k]->dz[l] = reinterpret_cast<float*>(take(rows * nets[k]->dims[l] * sizeof(float)));
        }
    }
    // act'(z) of every hidden layer, for activations whose derivative cannot be recovered from their output: carved
    // last, so every other buffer (and the workspace of the other activations) keeps its offset
    for (int k = 0; k < 2; ++k) {
        const bool stored = act_stores_derivative(nets[k]->activation);
        for (int l = 0; l <= PPOAF_MAX_LAYERS; ++l) ns[k]->dact[l] = nullptr;
        for (int l = 1; stored && l < nets[k]->n_layers; ++l)
            ns[k]->dact[l] = reinterpret_cast<float*>(take(size_t(max_batch) * nets[k]->dims[l] * sizeof(float)));
    }
    out->total = off;
}

int check_cfg(const ppoaf_update_cfg* cfg, const char* who) {
    PPOAF_CHECK_ARG(cfg != nullptr, "%s: null cfg", who);
    if (check_mlp_desc(&cfg->actor, who) || check_mlp_desc(&cfg->critic, who)) return 1;
    PPOAF_CHECK_ARG(cfg->critic.dims[cfg->critic.n_layers] == 1, "%s: critic output width must be 1", who);
    PPOAF_CHECK_ARG(cfg->head == PPOAF_HEAD_GAUSSIAN_TANH || cfg->head == PPOAF_HEAD_CATEGORICAL ||
                    cfg->head == PPOAF_HEAD_MULTI_CATEGORICAL || cfg->head == PPOAF_HEAD_BERNOULLI, "%s: unknown head", who);
    const int pred = cfg->actor.dims[cfg->actor.n_layers];
    if (cfg->head == PPOAF_HEAD_GAUSSIAN_TANH) {
        PPOAF_CHECK_ARG(pred == cfg->act_dim, "%s: Gaussian actor output width must equal act_dim", who);
        PPOAF_CHECK_ARG(pred <= kMaxGaussianDims, "%s: head width %d is outside the 1 .. %d dims of the Gaussian head",
                        who, pred, kMaxGaussianDims);
    } else if (cfg->head == PPOAF_HEAD_BERNOULLI) {
        PPOAF_CHECK_ARG(pred == cfg->act_dim,
                        "%s: Bernoulli actor output width must equal act_dim (one column per binary action)", who);
        PPOAF_CHECK_ARG(pred <= kMaxNarrowHead, "%s: head width %d is outside the 1 .. %d columns of the Bernoulli head",
                        who, pred, kMaxNarrowHead);
    } else if (cfg->head == PPOAF_HEAD_MULTI_CATEGORICAL) {
        PPOAF_CHECK_ARG(pred <= kMaxNarrowHead,
                        "%s: head width %d is outside the 1 .. %d outputs of the multi-categorical head", who, pred,
                        kMaxNarrowHead);
        PPOAF_CHECK_ARG(section_table_ok(cfg_section_ends(cfg), pred, cfg->act_dim),
                        "%s: bad multi-categorical section table (must be nonzero, its highest set bit must be the last "
                        "actor output, at most 64 outputs, and it must have act_dim = %d bits)", who, cfg->act_dim);
    } else {
        PPOAF_CHECK_ARG(cfg->act_dim == 1, "%s: Categorical actions are stored as one int64 index", who);
        PPOAF_CHECK_ARG(pred <= kMaxCategoricalClasses,
                        "%s: head width %d is outside the 1 .. %d classes of the Categorical head", who, pred,
                        kMaxCategoricalClasses);
    }
    return 0;
}

}  // namespace ppoaf

using namespace ppoaf;

extern "C" int ppoaf_abi_version(void) { return PPOAF_ABI_VERSION; }
extern "C" const char* ppoaf_last_error(void) { return g_err; }

extern "C" int ppoaf_device_info(int* sm, int* cc_major, int* cc_minor) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        set_error("ppoaf_device_info: no CUDA device: %s", cudaGetErrorString(e));
        return 1;
    }
    cudaDeviceProp p;
    e = cudaGetDeviceProperties(&p, dev);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_device_info: %s", cudaGetErrorString(e));
    if (sm) *sm = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return 0;
}

extern "C" int ppoaf_runtime_init(void) {
    int dev = 0;
    cudaError_t e0 = cudaGetDevice(&dev);
    PPOAF_CHECK_ARG(e0 == cudaSuccess, "ppoaf_runtime_init: no CUDA device: %s", cudaGetErrorString(e0));
    configure_gemm_kernels();
    configure_stats_kernels();
    cudaError_t e = cudaGetLastError();
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_runtime_init: %s", cudaGetErrorString(e));
    return 0;
}

extern "C" size_t ppoaf_update_workspace_bytes(const ppoaf_update_cfg* cfg, int32_t max_batch) {
    if (!cfg || max_batch <= 0) return 0;
    StepScratch s;
    carve(cfg, max_batch, nullptr, &s);
    return s.total;
}

#define PPOAF_CUDA_OK(expr, what)                                                      \
    do {                                                                               \
        cudaError_t e__ = (expr);                                                      \
        if (e__ != cudaSuccess) {                                                      \
            set_error("%s: %s", what, cudaGetErrorString(e__));                        \
            return 2;                                                                  \
        }                                                                              \
    } while (0)

#ifdef PPOAF_GEMM_TIMING
// debug build only: stop the chain after PPOAF_STOP_AFTER launches (prefix timing of the step, scratch/prefix_times.py)
#include <stdlib.h>
static int stop_after() { const char* e = getenv("PPOAF_STOP_AFTER"); return e ? atoi(e) : 1000; }
#define PPOAF_STEP_LIMIT() do { if (++launched__ > stop_after()) return 0; } while (0)
#else
#define PPOAF_STEP_LIMIT() do {} while (0)
#endif

extern "C" int ppoaf_ppo_minibatch_grads(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* b, void* stream) {
#ifdef PPOAF_GEMM_TIMING
    int launched__ = 0;
#endif
    if (check_cfg(cfg, "ppoaf_ppo_minibatch_grads")) return 1;
    PPOAF_CHECK_ARG(b != nullptr && b->batch >= 1 && b->batch <= b->batch_size && b->n_flat > 0,
                    "ppoaf_ppo_minibatch_grads: bad batch sizes");
    PPOAF_CHECK_ARG(b->n_mirror >= 0 && b->n_mirror <= PPOAF_MAX_MIRROR, "ppoaf_ppo_minibatch_grads: n_mirror out of range");
    if (b->batch == 1) return 0;  // the reference skips one-row minibatches (ppo.py:2305)
    PPOAF_CHECK_ARG(b->workspace_bytes >= ppoaf_update_workspace_bytes(cfg, b->batch_size),
                    "ppoaf_ppo_minibatch_grads: workspace too small");
    PPOAF_CHECK_ARG(reinterpret_cast<uintptr_t>(b->workspace) % 256 == 0,
                    "ppoaf_ppo_minibatch_grads: workspace must be 256-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;

    StepScratch sc;
    carve(cfg, b->batch_size, reinterpret_cast<char*>(b->workspace), &sc);  // layout fixed by the nominal B
    const bool gaussian = cfg->head == PPOAF_HEAD_GAUSSIAN_TANH;
    int64_t off[2][2 * PPOAF_MAX_LAYERS + 1];
    const int64_t n_actor = param_layout(&cfg->actor, gaussian ? cfg->act_dim : 0, off[0]);
    param_layout(&cfg->critic, 0, off[1]);
    const ppoaf_mlp_desc* net[2] = {&cfg->actor, &cfg->critic};
    const float* par[2] = {b->params, b->params + n_actor};
    float* grd[2] = {b->grads, b->grads + n_actor};
    const float* x0[2] = {b->obs, b->critic_obs};
    NetScratch* ns[2] = {&sc.actor, &sc.critic};
    const int L[2] = {cfg->actor.n_layers, cfg->critic.n_layers};
    const int Lmax = L[0] > L[1] ? L[0] : L[1];
    const int rows = b->batch;
    // The two head layers (last Linear of actor and critic) and their dX are computed inside the loss kernel when
    // their shapes allow it: two of the ten launches of the step disappear.
    const bool fuse_heads = L[0] == L[1] && L[0] >= 2 && cfg->actor.activation == cfg->critic.activation &&
                            getenv("PPOAF_NO_HEAD_FUSION") == nullptr &&
                            loss_head_fusable(cfg->actor.dims[L[0]], cfg->actor.dims[L[0] - 1],
                                              cfg->critic.dims[L[1] - 1], cfg->vf_clip_enabled);

    // ---- forward: layer l of both networks in one grouped launch ----
    for (int l = 0; l < Lmax - (fuse_heads ? 1 : 0); ++l) {
        GemmGroup grp(GEMM_BACKEND_FFMA);   // the update always runs the FFMA tiles: fp32 FMA accuracy (the stand-alone tcgen05 tiles keep one accumulator)
        for (int k = 0; k < 2; ++k) {
            if (l >= L[k]) continue;
            const bool first = l == 0, last = l + 1 == L[k];
            grp.add_forward(first ? x0[k] : ns[k]->act[l], net[k]->dims[l], first ? b->perm : nullptr,
                            par[k] + off[k][2 * l], par[k] + off[k][2 * l + 1], ns[k]->act[l + 1], rows,
                            net[k]->dims[l], net[k]->dims[l + 1], last ? PPOAF_ACT_IDENTITY : net[k]->activation,
                            /*w_static=*/l > 0, last ? nullptr : ns[k]->dact[l + 1]);
        }
        PPOAF_STEP_LIMIT();
        if (grp.launch(b->mb_cursor, b->batch_size, s)) return 2;
    }

    // ---- fused loss forward/backward ----
    LossArgs a{};
    a.actor_out = sc.actor.act[L[0]];
    a.critic_out = sc.critic.act[L[1]];
    a.log_std = gaussian ? par[0] + off[0][2 * L[0]] : nullptr;
    a.raw_actions = b->raw_actions;
    a.advantages = b->advantages;
    a.log_probs = b->log_probs;
    a.rewards_to_go = b->rewards_to_go;
    a.values = b->values;
    a.perm = b->perm;
    a.cursor = b->mb_cursor;
    a.batch_size = b->batch_size;
    a.batch = rows;
    a.mb_adv_stats = b->mb_adv_stats;
    a.mb_val_stats = b->mb_val_stats;
    a.hparams = b->hparams;
    a.epoch_stats = b->epoch_stats;
    a.d_actor_out = sc.actor.dz[L[0]];
    a.d_critic_out = sc.critic.dz[L[1]];
    a.d_log_std = gaussian ? grd[0] + off[0][2 * L[0]] : nullptr;
    a.sq_log_std = sc.sq_actor + (sc.n_sq_actor - 1);
    a.partials = sc.loss_partials;
    a.ticket = sc.loss_ticket;
    a.head = cfg->head;
    a.act_dim = cfg->act_dim;
    a.pred_dim = cfg->actor.dims[L[0]];
    a.section_ends = cfg_section_ends(cfg);
    a.use_huber = cfg->use_huber;
    a.normalize_adv = cfg->normalize_adv;
    a.normalize_values = cfg->normalize_values;
    a.vf_clip_enabled = cfg->vf_clip_enabled;
    a.min_std = cfg->min_std;
    a.pf_rows[0] = b->obs;
    a.pf_rows[1] = b->critic_obs;
    a.pf_row_bytes[0] = cfg->actor.dims[0] * int(sizeof(float));
    a.pf_row_bytes[1] = cfg->critic.dims[0] * int(sizeof(float));
    a.n_flat = b->n_flat;
    a.n_mirror = b->n_mirror;
    for (int q = 0; q < b->n_mirror; ++q) a.mirror_delta[q] = b->mirror_delta[q];
    a.fused = fuse_heads ? 1 : 0;
    if (fuse_heads) {
        a.h_actor = sc.actor.act[L[0] - 1];
        a.h_critic = sc.critic.act[L[1] - 1];
        a.W_actor = par[0] + off[0][2 * (L[0] - 1)];
        a.b_actor = par[0] + off[0][2 * (L[0] - 1) + 1];
        a.W_critic = par[1] + off[1][2 * (L[1] - 1)];
        a.b_critic = par[1] + off[1][2 * (L[1] - 1) + 1];
        a.dz_actor = sc.actor.dz[L[0] - 1];
        a.dz_critic = sc.critic.dz[L[1] - 1];
        a.dact_actor = sc.actor.dact[L[0] - 1];
        a.dact_critic = sc.critic.dact[L[1] - 1];
        a.Ha = cfg->actor.dims[L[0] - 1];
        a.Hc = cfg->critic.dims[L[1] - 1];
        a.act = cfg->actor.activation;
    }
    PPOAF_STEP_LIMIT();
    if (launch_ppo_loss(a, s)) return 2;

    // ---- backward: dW/db and dX of one layer of both networks per grouped launch, top layer first ----
    double* sq[2] = {sc.sq_actor, sc.sq_critic};
    int sq_used[2] = {0, 0};
    for (int k_top = fuse_heads ? 1 : 0; k_top < Lmax; ++k_top) {
        GemmGroup grp(GEMM_BACKEND_FFMA);   // the update always runs the FFMA tiles: fp32 FMA accuracy (the stand-alone tcgen05 tiles keep one accumulator)
        for (int k = 0; k < 2; ++k) {
            const int l = L[k] - 1 - k_top;
            if (l < 0) continue;
            const bool first = l == 0;
            if (fuse_heads && k_top == 1) {    // the heads' dW / db (their dX came out of the loss kernel)
                const int lh = L[k] - 1;
                sq_used[k] += grp.add_backward_w(ns[k]->dz[lh + 1], ns[k]->act[lh], net[k]->dims[lh], nullptr,
                                                 grd[k] + off[k][2 * lh], grd[k] + off[k][2 * lh + 1], rows,
                                                 net[k]->dims[lh], net[k]->dims[lh + 1], sq[k] + sq_used[k],
                                                 /*x_static=*/true);
            }
            sq_used[k] += grp.add_backward_w(ns[k]->dz[l + 1], first ? x0[k] : ns[k]->act[l], net[k]->dims[l],
                                             first ? b->perm : nullptr, grd[k] + off[k][2 * l],
                                             grd[k] + off[k][2 * l + 1], rows, net[k]->dims[l], net[k]->dims[l + 1],
                                             sq[k] + sq_used[k], /*x_static=*/!first);
            if (!first)
                grp.add_backward_x(ns[k]->dz[l + 1], par[k] + off[k][2 * l], ns[k]->dact[l] ? ns[k]->dact[l] : ns[k]->act[l],
                                   ns[k]->dz[l], rows, net[k]->dims[l], net[k]->dims[l + 1], net[k]->activation);
        }
        PPOAF_STEP_LIMIT();
        if (grp.launch(b->mb_cursor, b->batch_size, s, b->n_mirror, b->mirror_delta)) return 2;
    }
    return 0;
}

extern "C" int ppoaf_ppo_minibatch_apply(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* b, void* stream) {
    if (check_cfg(cfg, "ppoaf_ppo_minibatch_apply")) return 1;
    PPOAF_CHECK_ARG(b != nullptr && b->batch >= 1, "ppoaf_ppo_minibatch_apply: bad batch");
    cudaStream_t s = (cudaStream_t)stream;
    if (b->batch == 1) return launch_advance_cursor(b->mb_cursor, s);
    StepScratch sc;
    carve(cfg, b->batch_size, reinterpret_cast<char*>(b->workspace), &sc);
    const bool gaussian = cfg->head == PPOAF_HEAD_GAUSSIAN_TANH;
    const int64_t n_actor = param_layout(&cfg->actor, gaussian ? cfg->act_dim : 0, nullptr);
    const int64_t n_critic = param_layout(&cfg->critic, 0, nullptr);
    // Single rank: the backward-w epilogues already left the per-tile sums of squares.  R > 1: the caller has
    // all-reduced `grads` in between, so the norm must be taken again over the reduced buffer.
    const bool fused_norm = cfg->world_size <= 1;
    return launch_clip_adam(b->params, b->grads, b->adam_m, b->adam_v, b->adam_step, b->mb_cursor, b->hparams, n_actor,
                            n_critic, fused_norm ? sc.sq_actor : nullptr, sc.n_sq_actor,
                            fused_norm ? sc.sq_critic : nullptr, sc.n_sq_critic, sc.optim_ws, s,
                            /*chained=*/fused_norm);
}
