/*
 * ppoaf_b200.h — C ABI of libppoaf_b200.so: the B200 (sm_100a) implementation of the
 * PPO-AF post-rollout update path (LLNL/ppo_and_friends).
 *
 * The reference is pure Python and has no FFI of its own; its "plugin surface" for this
 * path is the duck-typed policy/dataset API (SURVEY.md §8b).  These entry points are what
 * a ctypes binding placed behind that API calls (INTEGRATION.md shows the binding).  Each
 * function names the reference code it replaces as file:line in /root/reference.
 *
 * Conventions
 *   - plain C types only; every pointer is a DEVICE pointer unless the name ends in _host;
 *   - no ownership transfer: the caller (torch) owns all memory, including workspaces whose
 *     size is obtained from the matching *_workspace_bytes() query;
 *   - `stream` is a cudaStream_t passed as void*; every call only ENQUEUES work on it and is
 *     legal during CUDA-graph stream capture (no allocation, no synchronisation);
 *   - return value 0 = success, nonzero = error; ppoaf_last_error() gives the message of the
 *     last failing call on the calling thread;
 *   - float data is fp32; running statistics and scan accumulation are fp64 on device.
 */
#ifndef PPOAF_B200_H
#define PPOAF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PPOAF_ABI_VERSION 1
#define PPOAF_MAX_LAYERS 8

/* activation ids (hidden layers of FeedForwardNetwork, networks/utils.py:160-183) */
enum { PPOAF_ACT_IDENTITY = 0, PPOAF_ACT_RELU = 1, PPOAF_ACT_LEAKY_RELU = 2, PPOAF_ACT_TANH = 3 };
/* action heads (networks/distributions.py).  PPOAF_HEAD_MULTI_CATEGORICAL (MultiDiscrete action spaces,
 * MultiCategoricalDistribution :272-438) is a restatement, not pinned by a reference golden: softmax over the whole
 * actor output row, then one torch Categorical(probs) per section of the row (renormalised, clamped to [eps, 1-eps]);
 * log-prob and entropy are the sums over the sections.  The sections are described by a 64-bit table of section
 * ends (bit c set: actor output c is the last of its section), so the row holds at most 64 outputs; nvec must be
 * 1-D with start = 0 and every entry >= 1.  PPOAF_HEAD_BERNOULLI (MultiBinary action spaces, BernoulliDistribution
 * :134-196) is a restatement too: one torch Bernoulli(probs = sigmoid(actor output)) per output column, log-prob and
 * entropy summed over the columns; act_dim = actor output width = number of columns (at most 64), fp32 0/1 actions.
 * Widths: PPOAF_HEAD_CATEGORICAL takes 1 .. 65536 classes and PPOAF_HEAD_GAUSSIAN_TANH 1 .. 4096 dimensions; rows of
 * more than 64 outputs run one CTA (update) or one warp (evaluation, sampling) per row instead of one warp / thread.
 * The multi-categorical and Bernoulli heads take at most 64 outputs.  Wider rows are refused, naming the width. */
enum { PPOAF_HEAD_GAUSSIAN_TANH = 0, PPOAF_HEAD_CATEGORICAL = 1, PPOAF_HEAD_MULTI_CATEGORICAL = 2, PPOAF_HEAD_BERNOULLI = 3 };

int         ppoaf_abi_version(void);
const char* ppoaf_last_error(void);
/* sm count / compute capability of the current device; fails (nonzero) when no CUDA device. */
int         ppoaf_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* One-time per-device setup (kernel attributes such as > 48 KB dynamic shared memory); call once
 * before the first stream capture. */
int         ppoaf_runtime_init(void);
/* Engine of ppoaf_mlp_forward's GEMMs: 0 = fp32 FFMA tiles (default), 1 = tcgen05 3xTF32 tensor-core tiles.
 * The update always runs the FFMA tiles (or the fused step's own tensor-core tiles, PPOAF_STEP=fused). */
int         ppoaf_set_gemm_backend(int backend);
int         ppoaf_get_gemm_backend(void);

/* ------------------------------------------------------------------------------------------
 * A2/A5  Segment table -> flat dataset order.
 * Replaces combine_episodes / PPODataset.add_episode ordering (utils/episode_info.py:44-135,
 * 701-719): segment s (in completion order) covers ring rows (t0[s] + k) * n_cols + col[s],
 * k < len[s], and lands at flat positions off[s] .. off[s]+len[s]-1.
 * Outputs: src_row[N] (ring row of each flat element), seg_flag[N] (bit0 = last element of a
 * segment, bit1 = that segment ended terminal).
 * ---------------------------------------------------------------------------------------- */
int ppoaf_build_flat_map(const int32_t* seg_col, const int32_t* seg_t0, const int32_t* seg_len,
                         const int64_t* seg_off, const uint8_t* seg_terminal, int32_t n_seg,
                         int32_t n_cols, int64_t n_flat, int32_t* src_row, uint8_t* seg_flag,
                         void* stream);

/* A5/A6/A7  Row gather  dst[i, :] = src[idx[i] * src_stride_bytes .. + row_bytes)  (src_stride_bytes = 0
 * means densely packed rows).  The strided form de-interleaves one field out of the packed
 * rollout ring, whose row holds every per-timestep field of one (step, env, agent).
 * Replaces the list->array->tensor copies of PPODataset.build (utils/episode_info.py:745-914)
 * and DataLoader collate of __getitem__ rows (utils/episode_info.py:916-987).  idx is int32
 * (idx_is_64 = 0) or int64 (idx_is_64 = 1, the minibatch permutation). */
int ppoaf_gather_rows(const void* src, int64_t src_stride_bytes, const void* idx, int idx_is_64, void* dst,
                      int64_t n_rows, int64_t row_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * A3/A4/P7  GAE + reward-to-go as ONE segmented reverse scan over the flattened buffer.
 * Replaces EpisodeInfo.end_episode / compute_discounted_sums / _compute_gae_advantages /
 * _compute_standard_advantages (utils/episode_info.py:223-301, 401-465) and
 * PPODataset.recalculate_advantages (:721-743).
 *   rewards, values  fp32 [N] in flat order;  seg_flag [N] from ppoaf_build_flat_map;
 *   seg_off int64 [n_seg+1] flat offsets;  v_boot, r_boot fp32 [n_seg] per-segment seeds
 *   (r_boot already clipped to bootstrap_clip, SURVEY Q2);  use_gae = 0 -> adv = rtg - V.
 *   Accumulation is fp64, outputs fp32.  Algorithmic traffic 17 B/timestep + 9 B/segment.
 * ---------------------------------------------------------------------------------------- */
size_t ppoaf_segscan_workspace_bytes(int64_t n_flat);
int ppoaf_gae_rtg_segscan(const float* rewards, const float* values, const uint8_t* seg_flag,
                          const int64_t* seg_off, const float* v_boot, const float* r_boot,
                          int32_t n_seg, int64_t n_flat, double gamma, double lambd, int use_gae,
                          float* adv_out, float* rtg_out, void* workspace, size_t workspace_bytes,
                          void* stream);

/* ------------------------------------------------------------------------------------------
 * N1  RunningMeanStd.update (utils/stats.py:29-94): column moments of x[n_rows, dim] and the
 * Chan merge into the running state.  state = fp64 [2*dim + 1] = mean[dim] | var[dim] | count.
 *   ppoaf_batch_moments  writes the batch triple fp64 [2*dim+1] = mean | M2 | n  (no merge), so
 *                        that triples of several ranks can be exchanged and merged in rank order;
 *   ppoaf_stats_merge    merges n_triples batch triples (concatenated) into `state`, pooling
 *                        them first exactly like the reference's allgather+concatenate (:47-53).
 * ---------------------------------------------------------------------------------------- */
size_t ppoaf_moments_workspace_bytes(int64_t n_rows, int32_t dim);
int ppoaf_batch_moments(const float* x, int64_t n_rows, int32_t dim, double* triple_out,
                        void* workspace, size_t workspace_bytes, void* stream);
int ppoaf_stats_merge(double* state, const double* triples, int32_t n_triples, int32_t dim,
                      void* stream);

/* N2/N4  y = clip((x - mean) / sqrt(var + eps), lo, hi) over x[n_rows, dim]  (utils/misc.py:106-111,
 * environments/filter_wrappers.py:220-221, 655-657).  lo >= hi disables the clip.  In-place ok.
 * ppoaf_denormalize: y = mean + x * sqrt(var + eps) (utils/misc.py:124-128). */
int ppoaf_normalize_clip(const float* x, int64_t n_rows, int32_t dim, const double* state, float eps,
                         float lo, float hi, float* y, void* stream);
int ppoaf_denormalize(const float* x, int64_t n_rows, int32_t dim, const double* state, float eps,
                      float* y, void* stream);

/* "Next" row 2 (SURVEY §8f): the reward normaliser's environment step, RewardNormalizer.step
 * (environments/filter_wrappers.py:393-425) with its sequential-in-time semantics (SURVEY Q9): running_reward[e] =
 * running_reward[e] * gamma + rewards[e] for e = 0 .. E-1 IN ORDER, the whole partially updated vector entering the running
 * statistics after every element.  ppoaf_reward_norm_triples writes the E batch triples (mean | M2 | n) of one step and
 * zeroes running_reward where `dones`; the caller all-gathers them across ranks and integrates them with
 * ppoaf_value_stats_sequence (n_mb = E), which pools the ranks per element exactly like the reference's allgather.
 * ppoaf_reward_scale_clip: y = clip(r / sqrt(var + eps), lo, hi)  (:466-476, RewardClipper :700-719; lo >= hi: no clip). */
int ppoaf_reward_norm_triples(const float* rewards, const uint8_t* dones, double* running_reward /* fp64 [E], in/out */,
                              int32_t n_envs, double gamma, double* triples_out /* fp64 [E, 3] */, void* stream);
int ppoaf_reward_scale_clip(const float* rewards, const double* state /* fp64 [3]: mean, var, count */, float eps,
                            float lo, float hi, float* out, int32_t n, void* stream);

/* ------------------------------------------------------------------------------------------
 * P1..P4  The minibatch update.
 * ---------------------------------------------------------------------------------------- */
typedef struct {
    int32_t n_layers;                       /* number of Linear layers (hidden_depth + 1)          */
    int32_t dims[PPOAF_MAX_LAYERS + 1];     /* in, h1, ..., out                                    */
    int32_t activation;                     /* PPOAF_ACT_* for hidden layers                       */
} ppoaf_mlp_desc;

/* hyper-parameters live in a DEVICE fp64 block (python floats are doubles; kernels round to fp32 where torch does) read by the kernels each step (SURVEY row P8),
 * so schedulers can change them between graph replays without re-capturing. */
enum {
    PPOAF_HP_LR = 0, PPOAF_HP_ENTROPY_WEIGHT, PPOAF_HP_SURR_CLIP, PPOAF_HP_GRAD_CLIP /* <0: off */,
    PPOAF_HP_KL_WEIGHT, PPOAF_HP_VF_CLIP /* <0: off */, PPOAF_HP_BETA1, PPOAF_HP_BETA2,
    PPOAF_HP_ADAM_EPS, PPOAF_HP_INV_WORLD /* 1/R applied to summed grads */, PPOAF_HP_COUNT = 16
};
/* per-epoch statistics, DEVICE fp64 block (ppo.py:2280-2285, 2471-2485) */
enum {
    PPOAF_ST_ACTOR_LOSS = 0, PPOAF_ST_CRITIC_LOSS, PPOAF_ST_ENTROPY, PPOAF_ST_KL, PPOAF_ST_COUNTER,
    PPOAF_ST_BAD_RATIO /* nan/inf ratios seen (ppo.py:2361) */, PPOAF_ST_BAD_VALUE /* nan in nets */,
    PPOAF_ST_COUNT = 8
};

typedef struct {
    ppoaf_mlp_desc actor, critic;
    int32_t head;                 /* PPOAF_HEAD_*                                                    */
    int32_t act_dim;              /* stored action width: Da (Gaussian, 1 .. 4096), 1 (Categorical
                                     index, 1 .. 65536 classes), the number of sections
                                     (Multi-categorical, one int64 index each) or the number of
                                     columns (Bernoulli, = actor output width); the last two <= 64   */
    int32_t use_huber;            /* nn.HuberLoss(delta=10) instead of MSE (ppo.py:2416-2419)       */
    int32_t normalize_adv;        /* ppo.py:2325-2333                                               */
    int32_t normalize_values;     /* ppo.py:2299-2303                                               */
    int32_t vf_clip_enabled;      /* value clip on (clip value itself is PPOAF_HP_VF_CLIP)          */
    int32_t world_size;           /* ranks whose gradients the caller all-reduces between grads/apply */
    int32_t reserved[1];
    float   min_std;              /* GaussianDistribution min_std (networks/distributions.py:453)   */
    uint32_t section_ends[2];     /* Multi-categorical section table, 64-bit mask (lo, hi): bit c set =
                                     actor output c ends a section.  Nonzero, highest bit = outputs - 1,
                                     popcount = act_dim.  Read by no other head (leave it zero).      */
    float   reserved_f[1];
} ppoaf_update_cfg;

/* Flat parameter layout (shared by params / grads / Adam m / Adam v): for each net, for each
 * layer W[out,in] row-major then b[out], in the reference's parameters() order; the Gaussian
 * actor appends log_std[act_dim] (distribution.log_std).  Every tensor starts on a 4-float
 * boundary.  Layout: [actor | critic].  ppoaf_param_layout fills offsets (in floats):
 *   offsets[2*l] = W_l, offsets[2*l+1] = b_l, then log_std (actor only); returns total floats. */
int64_t ppoaf_param_layout(const ppoaf_mlp_desc* net, int32_t log_std_dim, int64_t* offsets /* [2*L+1] */);

#define PPOAF_MAX_MIRROR 7      /* peers a rank can push its gradients to (R <= 8) */
typedef struct {
    /* dataset in flat order (PPODataset attributes, utils/episode_info.py:823-912) */
    const float*   critic_obs;    /* [N, Dc] */
    const float*   obs;           /* [N, Do] */
    const void*    raw_actions;   /* [N, act_dim] fp32 (Gaussian, Bernoulli 0/1) or int64 (Categorical) */
    const float*   advantages;    /* [N] */
    const float*   log_probs;     /* [N] */
    const float*   rewards_to_go; /* [N] */
    float*         values;        /* [N]  overwritten with critic outputs (ppo.py:2340) */
    const int64_t* perm;          /* [N]  this epoch's permutation (RandomSampler protocol, row U1) */
    /* per-epoch minibatch tables from ppoaf_epoch_prepare */
    const float*   mb_adv_stats;  /* [n_mb, 2] mean, 1/(std_unbiased + 1e-8) */
    const float*   mb_val_stats;  /* [n_mb, 2] mean, 1/sqrt(var + 1e-8) AFTER integrating minibatch k */
    /* networks: flat [actor | critic] */
    float* params; float* grads; float* adam_m; float* adam_v;
    int64_t* adam_step;           /* device scalar t */
    const double* hparams;        /* [PPOAF_HP_COUNT] */
    double* epoch_stats;          /* [PPOAF_ST_COUNT] */
    int32_t* mb_cursor;           /* device scalar: index of the minibatch to run; advanced by _apply */
    void* workspace; size_t workspace_bytes;
    int64_t n_flat;               /* N */
    int32_t batch;                /* rows in THIS minibatch (== batch_size except the last one) */
    int32_t batch_size;           /* nominal B: minibatch k covers perm[k*B .. k*B+batch) */
    /* R > 1, push exchange: every gradient element written to `grads` is also stored at
     * (char*)address + mirror_delta[q] for q < n_mirror — the slot this rank owns inside every peer's receive
     * buffer (peer memory mapped with ppoaf_peer_import), so the gradients cross NVLink while the backward pass
     * is still running.  n_mirror == 0: local gradients only. */
    int32_t n_mirror;
    int32_t reserved0;
    int64_t mirror_delta[PPOAF_MAX_MIRROR];
} ppoaf_update_bufs;

size_t ppoaf_update_workspace_bytes(const ppoaf_update_cfg* cfg, int32_t max_batch);

/* Once per epoch, from (perm, advantages, rewards_to_go): per-minibatch advantage mean / unbiased
 * std (ppo.py:2325-2333) and per-minibatch reward-to-go triples for the value normaliser
 * (ppo.py:2299-2303 -> utils/misc.py:100-104 -> utils/stats.py:29-59).  mb_val_triples fp64
 * [n_mb, 3] = mean | M2 | n can be all-gathered across ranks; ppoaf_value_stats_sequence then
 * integrates them in (minibatch, rank) order into `state` (fp64 [3]: mean, var, count) and writes
 * mb_val_stats[k].  Minibatches of one row still update the statistics (the reference normalises
 * before its skip test, ppo.py:2299-2306). */
int ppoaf_epoch_prepare(const int64_t* perm, const float* advantages, const float* rewards_to_go,
                        int64_t n_flat, int32_t batch_size, float* mb_adv_stats,
                        double* mb_val_triples, void* stream);
int ppoaf_value_stats_sequence(double* state, const double* mb_val_triples /* [n_ranks, n_mb, 3] */,
                               int32_t n_ranks, int32_t n_mb, float eps, float* mb_val_stats,
                               void* stream);

/* One minibatch, first half: gather -> actor & critic forward (policies/ppo_policy.py:891-952,
 * networks/ppo_networks/feed_forward.py:66-86) -> fused loss forward/backward (ppo.py:2342-2438)
 * -> backward into `grads` (this rank's local gradient).
 * Second half (after the caller's all-reduce of `grads` when R > 1): grads *= 1/R
 * (utils/mpi_utils.py:89-111), per-net clip_grad_norm_ and Adam (policies/ppo_policy.py:1032-1055),
 * then advances mb_cursor and adam_step. */
int ppoaf_ppo_minibatch_grads(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* bufs, void* stream);
int ppoaf_ppo_minibatch_apply(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* bufs, void* stream);

/* The same minibatch step(s) as ONE persistent launch (fused_step.cu): n_steps consecutive minibatches of bufs->batch rows,
 * starting at *mb_cursor, each = forward (TMA boxes + tcgen05 3xTF32 tiles) -> heads + loss -> backward -> clip + Adam, the phases
 * separated by grid barriers instead of launch boundaries; mb_cursor and adam_step advance by n_steps.  Replaces the loop
 * body of PPO._ppo_batch_train (ppo.py:2292-2468) for a whole epoch.  Supported when ppoaf_ppo_fused_supported(cfg) != 0
 * (equal depth >= 2 and activation of actor and critic, head layers fusable into the loss phase: hidden width <= 256 and
 * a multiple of 4, <= 24 actor outputs, no value clipping; single rank); other configurations use
 * ppoaf_ppo_minibatch_grads / _apply.  Workspace: ppoaf_ppo_fused_workspace_bytes, zero-initialised once (it holds the
 * grid-barrier words, which persist from launch to launch).  n_steps > 1 requires bufs->batch == bufs->batch_size. */
int    ppoaf_ppo_fused_supported(const ppoaf_update_cfg* cfg);
size_t ppoaf_ppo_fused_workspace_bytes(const ppoaf_update_cfg* cfg, int32_t max_batch);
int    ppoaf_ppo_fused_steps(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* bufs, int32_t n_steps, void* stream);

/* Forward only (P1/P2; also rollout-time inference, SURVEY §8f row 1): y = MLP(x[idx]) for
 * n_rows rows; idx may be NULL (identity).  softmax applied when `softmax_out` (Discrete actor,
 * networks/distributions.py:1045); rows of more than 64 columns take a warp per row, whose sums run in a
 * different order than the one-thread-per-row kernel of narrower rows. */
size_t ppoaf_mlp_forward_workspace_bytes(const ppoaf_mlp_desc* net, int32_t n_rows);
int ppoaf_mlp_forward(const ppoaf_mlp_desc* net, const float* params, const float* x, const int64_t* idx,
                      int32_t n_rows, int softmax_out, float* y, void* workspace, size_t workspace_bytes,
                      void* stream);

/* P1  Action-head evaluation on its own (policies/ppo_policy.py:939-950): log-prob of `actions`
 * and entropy under the head parameterised by actor_out [n_rows, pred] (+ log_std for the
 * Gaussian head).  Widths (pred_dim and act_dim): Gaussian <= 4096, Categorical <= 65536, Bernoulli <= 64.  actions: fp32 [n_rows, act_dim] raw (pre-tanh), int64 [n_rows, 1] (Categorical) or
 * fp32 0/1 [n_rows, act_dim] (Bernoulli: actor_out holds the logits, pred = act_dim, log_std must be NULL;
 * log-prob and entropy are summed over the columns). */
int ppoaf_head_evaluate(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                        float min_std, const void* actions, int32_t act_dim, int32_t n_rows,
                        float* log_prob_out, float* entropy_out, void* stream);

/* "Next" row 1 (SURVEY §8f): rollout-time sampling, PPOPolicy.get_rollout_actions (policies/ppo_policy.py:729-794,
 * networks/distributions.py:518-655, 199-249).  `noise` holds the draws of the HOST generator in the order the reference's
 * CPU sampling consumes them -- N(0,1) [n_rows, act_dim] for the Gaussian head, Exp(1) [n_rows, pred_dim] for the
 * Categorical head (aten multinomial's one-sample path), U[0,1) [n_rows, act_dim] for the Bernoulli head (torch.rand,
 * as Bernoulli(probs).sample() draws it) -- so the sampled actions are the reference's.  Outputs:
 * raw_action / action fp32 [n_rows, act_dim] (Gaussian; action = tanh(raw) mapped to [dist_min, dist_max] when given),
 * int64 [n_rows, 1] (Categorical) or fp32 0/1 [n_rows, act_dim] (Bernoulli: action = [u < sigmoid(actor_out)], both
 * outputs get the same actions, each may be NULL; pred = act_dim; log_std, dist_min and dist_max must be NULL; noise of
 * 0.5 everywhere gives the deterministic action [p > 0.5]), log_prob fp32 [n_rows] (summed over the Bernoulli columns).
 * The Categorical head samples from softmax probs in actor_out.  Widths as for ppoaf_head_evaluate. */
int ppoaf_head_sample(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std, float min_std,
                      const float* noise, const float* dist_min, const float* dist_max, int32_t act_dim,
                      int32_t n_rows, void* raw_action_out, void* action_out, float* log_prob_out, void* stream);

/* The multi-categorical head (PPOAF_HEAD_MULTI_CATEGORICAL) on its own; (section_ends_lo, section_ends_hi) is the
 * section table of ppoaf_update_cfg.section_ends, n_sections its popcount.
 * _evaluate: log-prob of actions_i64 [n_rows, n_sections] (index inside each section) and entropy, from the actor's
 *   logits actor_out [n_rows, pred_dim] (PPOPolicy.evaluate).
 * _sample: rollout-time sampling from probs [n_rows, pred_dim] (ppoaf_mlp_forward with softmax_out = 1).  `noise` holds
 *   the host generator's Exp(1) draws in the order per-section Categorical sampling consumes them: section after
 *   section, a contiguous [n_rows, n_k] block each, so section k starting at output o_k reads
 *   noise[n_rows * o_k + i * n_k + j].  In each section a_k = first argmax(p~_k / q_k) (aten multinomial's one-sample
 *   path).  Outputs actions_out_i64 [n_rows, n_sections] and the summed log-prob [n_rows]. */
int ppoaf_multi_categorical_evaluate(const float* actor_out, int32_t pred_dim, uint32_t section_ends_lo,
                                     uint32_t section_ends_hi, const int64_t* actions_i64, int32_t n_sections,
                                     int32_t n_rows, float* log_prob_out, float* entropy_out, void* stream);
int ppoaf_multi_categorical_sample(const float* probs, int32_t pred_dim, uint32_t section_ends_lo,
                                   uint32_t section_ends_hi, const float* noise, int32_t n_sections, int32_t n_rows,
                                   int64_t* actions_out_i64, float* log_prob_out, void* stream);

/* ------------------------------------------------------------------------------------------
 * P5  Gradient all-reduce over NVLink peer memory FUSED with clip + Adam (R > 1 on one node).
 * Replaces mpi_avg_gradients (utils/mpi_utils.py:89-111) + clip_grad_norm_ + Adam.step
 * (policies/ppo_policy.py:1032-1055) with ONE kernel per rank: cross-GPU flag barrier, one-shot
 * reduce of the R peer gradient buffers in rank order (bit-identical on every rank), gradient norm,
 * clip, Adam.  Buffers come from ppoaf_peer_alloc (cudaMalloc) and are shared with CUDA IPC
 * handles that the host exchanges through torch.distributed; gradients are double-buffered by step
 * parity so one barrier per step suffices.  `ctrl`: local zeroed scratch of ppoaf_peer_ctrl_bytes().
 * ---------------------------------------------------------------------------------------- */
int    ppoaf_peer_alloc(size_t bytes, void** out);
int    ppoaf_peer_free(void* p);
int    ppoaf_peer_export(void* p, uint8_t* handle64);
int    ppoaf_peer_import(const uint8_t* handle64, void** out);
int    ppoaf_peer_close(void* p);
size_t ppoaf_peer_ctrl_bytes(void);
int    ppoaf_peer_allreduce_adam(const void* const* peer_grads, void* const* peer_flags, int32_t n_ranks,
                                 int32_t my_rank, float* params, float* adam_m, float* adam_v,
                                 int64_t* adam_step, int32_t* mb_cursor, const double* hparams,
                                 int64_t n_actor, int64_t n_critic, void* ctrl, void* stream);

/* P5, NVSwitch multicast (NVLS) variant: two-shot all-reduce fused with clip + Adam.  Gradient buffers, a parameter
 * staging buffer and one flag block per rank live in SYMMETRIC memory (torch.distributed._symmetric_memory provides the
 * peer and multicast mappings).  Rank r owns slice r of the flat parameters: multimem.ld_reduce returns the in-switch
 * sum of its slice, the slice norms are exchanged through the flag blocks, the owner applies clip + Adam (m, v are only
 * maintained for the owned slice) and stores the new parameters in its staging buffer; every rank then gathers all slices
 * from their owners' staging buffers (staging[r], peer mappings).  ~2 x 4 B/parameter of NVLink traffic per rank and
 * step, independent of R. */
size_t ppoaf_nvls_ctrl_bytes(void);
size_t ppoaf_nvls_flag_block_bytes(void);
int    ppoaf_nvls_allreduce_adam(const float* g_mc, void* const* staging, void* const* flag_blocks,
                                 int32_t n_ranks, int32_t my_rank, float* params, float* adam_m, float* adam_v,
                                 int64_t* adam_step, int32_t* mb_cursor, const double* hparams, int64_t n_actor,
                                 int64_t n_critic, void* ctrl, void* stream);

/* Stand-alone pieces (unit-parity entry points; the composite calls the same kernels). */
int ppoaf_clip_adam_step(float* params, const float* grads, float* adam_m, float* adam_v,
                         int64_t* adam_step, const double* hparams, int64_t n_actor, int64_t n_critic,
                         void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPOAF_B200_H */
