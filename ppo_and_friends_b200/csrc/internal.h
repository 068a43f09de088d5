// Internal (non-ABI) prototypes shared between the translation units of libppoaf_b200.so.
#pragma once
#include "common.cuh"

namespace ppoaf {

// mlp.cu — grouped GEMM launches (all GEMMs of one phase of the minibatch step in ONE launch)
enum { GEMM_BACKEND_FFMA = 0, GEMM_BACKEND_TCGEN05 = 1 };
int gemm_backend();             // PPOAF_GEMM=ffma|tcgen05 (default ffma); selects forward-only launches, see umma.cuh
struct GroupedGemmArgs;
constexpr int kMaxGroupHost = 6;    // problems one grouped launch carries (== kMaxGroup of mlp.cuh)
struct GemmGroup {
    GroupedGemmArgs* args;      // owned
    int n_tiles;
    int backend;
    explicit GemmGroup(int backend);
    ~GemmGroup();
    GemmGroup(const GemmGroup&) = delete;
    GemmGroup& operator=(const GemmGroup&) = delete;
    // Y[rows, out] = act(X[idx][rows, in] W^T + b); dact (FFMA tiles, act_stores_derivative ids): act'(z) [rows, out]
    // w_static / x_static: the operand is not written by the launch that precedes this one in the stream, so the
    // FFMA kernel may stage it before its programmatic-dependency wait (see common.cuh, PDL)
    void add_forward(const float* X, int ldx, const int64_t* idx, const float* W, const float* b, float* Y, int rows,
                     int in, int out, int act, bool w_static = false, float* dact = nullptr);
    // dX[rows, in] = (dZ[rows, out] W[out, in]) * act'(Xact[rows, in]); act_stores_derivative ids: Xact is act'(z)
    void add_backward_x(const float* dZ, const float* W, const float* Xact, float* dX, int rows, int in, int out, int act);
    // dW[out, in] = dZ[rows, out]^T X[idx][rows, in]; db[out] = column sums of dZ; sq_out[tile] = tile sum of squares
    // returns the number of sum-of-squares slots (tiles) this problem writes
    // (backward problems run on the FFMA tiles only: launch() refuses them in a GEMM_BACKEND_TCGEN05 group)
    int add_backward_w(const float* dZ, const float* X, int ldx, const int64_t* idx, float* dW, float* db, int rows,
                       int in, int out, double* sq_out, bool x_static = false);
    // n_mirror / mirror_delta: peer copies of the gradient buffer (ppoaf_update_bufs), applied to backward-w outputs
    int launch(const int32_t* cursor, int cursor_stride, cudaStream_t s, int n_mirror = 0,
               const int64_t* mirror_delta = nullptr);
};
int backward_w_tiles(int in, int out);
void configure_gemm_kernels();
int64_t param_layout(const ppoaf_mlp_desc* net, int32_t log_std_dim, int64_t* offsets);
int check_mlp_desc(const ppoaf_mlp_desc* net, const char* who);

// stats.cu — opts the column-moments kernel into the shared memory of its widest plan
void configure_stats_kernels();

// loss.cu
struct LossArgs {
    const float* actor_out;      // [batch, pred]  mean (Gaussian) or logits (Categorical)
    const float* critic_out;     // [batch]
    const float* log_std;        // [act_dim] (Gaussian)
    const void* raw_actions;     // dataset [N, act_dim] fp32 or int64
    const float* advantages;     // dataset [N]
    const float* log_probs;      // dataset [N]
    const float* rewards_to_go;  // dataset [N]
    float* values;               // dataset [N] (scatter target)
    const int64_t* perm;
    const int32_t* cursor;
    int batch_size;              // cursor stride
    int batch;                   // rows in this minibatch
    const float* mb_adv_stats;
    const float* mb_val_stats;
    const double* hparams;
    double* epoch_stats;
    float* d_actor_out;          // [batch, pred]
    float* d_critic_out;         // [batch]  (or [2, batch] scratch when vf_clip is on)
    float* d_log_std;            // [act_dim] inside grads
    double* sq_log_std;          // one slot: sum of squares of d_log_std (nullable)
    float* partials;             // workspace
    unsigned int* ticket;        // zero-initialised, self-resetting
    int head, act_dim, pred_dim;
    unsigned long long section_ends;   // PPOAF_HEAD_MULTI_CATEGORICAL: bit c set = actor output c ends a section
    int use_huber, normalize_adv, normalize_values, vf_clip_enabled;
    float min_std;
    // fused head layers (loss_head_fusable): the last Linear of both networks and its dX are computed by the loss
    // kernel itself, so actor_out / critic_out are not read and two GEMM launches disappear from the step
    int fused;
    const float* h_actor;        // [batch, Ha] activations below the actor head
    const float* h_critic;       // [batch, Hc]
    const float* W_actor;        // [pred, Ha]
    const float* b_actor;        // [pred]
    const float* W_critic;       // [1, Hc]
    const float* b_critic;       // [1]
    float* dz_actor;             // [batch, Ha]  dL/d(pre-activation of the layer below the head)
    float* dz_critic;            // [batch, Hc]
    const float* dact_actor;     // act_stores_derivative ids: act'(z) below the heads, [batch, Ha] / [batch, Hc]; else null
    const float* dact_critic;
    int Ha, Hc, act;
    int n_mirror;                // peer copies of d_log_std (push exchange)
    long long mirror_delta[PPOAF_MAX_MIRROR];
    // optional L2 prefetch of the next minibatch's gathered rows (obs, critic obs); pf_rows[0] == null: off
    const void* pf_rows[2];
    int pf_row_bytes[2];
    int64_t n_flat;
    // fused_step.cu: row pitch of d_actor_out / d_critic_out (0: dense, pred_dim / 1) - padded to 16 bytes there so that the
    // head layers' dW operand is a TMA-able matrix
    int d_actor_ld, d_critic_ld;
};
bool loss_head_fusable(int pred_dim, int Ha, int Hc, int vf_clip_enabled);
// Head widths.  Every head runs rows of up to kMaxNarrowHead actor outputs on the warp-per-sample kernels
// (loss_common.cuh); the Categorical and Gaussian heads also take wider rows, up to the bounds below, on the wide
// kernels of loss.cu.
constexpr int kMaxNarrowHead = 64;
constexpr int kMaxCategoricalClasses = 65536;
constexpr int kMaxGaussianDims = 4096;
// a multi-categorical section table that fits the row: nonzero, last section ends at pred_dim - 1, n_sections ends
bool section_table_ok(unsigned long long section_ends, int pred_dim, int n_sections);
// The Categorical head up to 64 classes is the table of one section (its callers leave cfg->section_ends zero); wider
// rows have no table: they run the wide loss kernel.
inline unsigned long long cfg_section_ends(const ppoaf_update_cfg* cfg) {
    if (cfg->head == PPOAF_HEAD_CATEGORICAL) {
        const int pred_dim = cfg->actor.dims[cfg->actor.n_layers];
        return pred_dim <= 64 ? 1ull << (pred_dim - 1) : 0ull;
    }
    return (uint64_t(cfg->section_ends[1]) << 32) | cfg->section_ends[0];
}
// step.cu: validates an update configuration (networks, head, section table); 0 = ok
int check_cfg(const ppoaf_update_cfg* cfg, const char* who);
size_t loss_workspace_bytes(int max_batch, int act_dim);
int launch_ppo_loss(const LossArgs& a, cudaStream_t s);

// optim.cu
// beta^t for the Adam bias corrections without a double pow() on the critical path: cache = (t, b1, b2, b1^t, b2^t) of
// the previous step; one multiply when t advanced by one under the same betas, pow() otherwise (first step, restored
// checkpoints, betas changed between steps, or a workspace shared by parameter sets with different betas).
constexpr int kBetaCacheDoubles = 5;
__device__ __forceinline__ void beta_powers(const double* cache, int64_t t, double b1, double b2, double& p1, double& p2) {
    if (cache[0] == double(t - 1) && t > 1 && cache[1] == b1 && cache[2] == b2) { p1 = cache[3] * b1; p2 = cache[4] * b2; }
    else { p1 = pow(b1, double(t)); p2 = pow(b2, double(t)); }
}
__device__ __forceinline__ void store_beta_powers(double* cache, int64_t t, double b1, double b2, double p1, double p2) {
    cache[0] = double(t); cache[1] = b1; cache[2] = b2; cache[3] = p1; cache[4] = p2;
}
// torch clip_grad_norm_'s coefficient for one network: max_norm / (norm + 1e-6) clamped to at most 1, with
// norm = sqrt(sumsq) * scale.  A NaN norm gives a NaN coefficient (torch.clamp keeps NaN), so a NaN gradient element
// makes every gradient of that network NaN, as in torch.  max_norm < 0: clipping off.
__device__ __forceinline__ float clip_coef(float max_norm, double sumsq, double scale) {
    if (!(max_norm >= 0.f)) return 1.f;
    const float c = max_norm / (float(sqrt(sumsq) * scale) + 1e-6f);
    return isnan(c) ? c : fminf(c, 1.f);
}
size_t optim_workspace_bytes();
// sq_a / sq_c: per-network sum-of-squares slots already produced by the backward-w epilogues (n_sq_* > 0), or
// null -> a norm pass over the (all-reduced) gradients is run first.
int launch_clip_adam(float* params, const float* grads, float* m, float* v, int64_t* adam_step, int32_t* mb_cursor,
                     const double* hparams, int64_t n_actor, int64_t n_critic, const double* sq_a, int n_sq_a,
                     const double* sq_c, int n_sq_c, void* workspace, cudaStream_t s, bool chained);
int launch_advance_cursor(int32_t* mb_cursor, cudaStream_t s);

}  // namespace ppoaf
