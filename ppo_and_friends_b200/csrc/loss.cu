// Fused PPO loss, forward + backward, for one minibatch (reference ppo.py:2299-2438 with the
// distribution arithmetic of networks/distributions.py:491-558,694 and torch's Normal/Categorical/Bernoulli).
// One WARP per sample (each lane owns action dims l, l + 32 and 8 hidden columns); nothing but the gradients w.r.t. the two network outputs, d(log_std) and
// six scalars ever reaches HBM.  Reductions are deterministic: per-CTA partials in fp64, summed in
// CTA order by the last CTA to finish (self-resetting ticket).
//
//   A^   = (A - mean_mb) / (std_mb + 1e-8)                        (mean/std precomputed per epoch)
//   rho  = exp(lp - lp_old);  L_actor = mean(-min(rho A^, clamp(rho, 1-eps, 1+eps) A^)) - w_H mean(H)
//   R^   = (RTG - mu_v) / sqrt(var_v + 1e-8);  L_critic = mean((v - R^)^2) | Huber(delta=10) [| value clip]
//   KL   = mean(lp_old - lp)  (statistic only: as a loss term it is a constant, SURVEY Q7)
#include "loss_common.cuh"

namespace ppoaf {

bool section_table_ok(unsigned long long section_ends, int pred_dim, int n_sections) {
    return pred_dim >= 1 && pred_dim <= kMaxAct && section_ends != 0 && 63 - __builtin_clzll(section_ends) == pred_dim - 1 &&
           __builtin_popcountll(section_ends) == n_sections;
}

bool loss_head_fusable(int pred_dim, int Ha, int Hc, int vf_clip_enabled) {
    auto ok = [](int H) { return H % 4 == 0 && H >= 4 && H <= 4 * kG * kFusedMaxChunks; };
    return pred_dim <= kFusedMaxPred && ok(Ha) && ok(Hc) && !vf_clip_enabled;
}


#ifdef PPOAF_GEMM_TIMING
__device__ long long g_loss_stamps[16];
#define LOSS_STAMP(k) do { if (threadIdx.x == 0 && (blockIdx.x == 0 || (k) >= 8)) g_loss_stamps[k] = clock64() - t_entry; } while (0)
#else
#define LOSS_STAMP(k) do {} while (0)
#endif

struct CtaBarrier { __device__ __forceinline__ void operator()() const { __syncthreads(); } };

template <bool FUSED>
__global__ void __launch_bounds__(kLossThreads) ppo_loss_kernel(const LossArgs a) {
    extern __shared__ __align__(16) float s_dyn[];      // FUSED: HeadSmem
    __shared__ float s_sd[kMaxAct], s_dsd[kMaxAct];
    __shared__ double s_red[kLossThreads / 32][kPartialStride];
    __shared__ double s_tot[kPartialStride];
    __shared__ double s_sq[kLossThreads / 32];
    __shared__ bool s_last;

#ifdef PPOAF_GEMM_TIMING
    const long long t_entry = clock64();
#endif
    const int tid = threadIdx.x;
    const int gl = tid & (kG - 1);                                   // lane inside the sample group
    const int i = blockIdx.x * kSamplesPerBlock + tid / kG;          // sample of this group
    const bool live = i < a.batch;
    const float inv_b = 1.0f / float(a.batch);
    const float w_ent = float(a.hparams[PPOAF_HP_ENTROPY_WEIGHT]);
    const float clip_lo = float(1.0 - a.hparams[PPOAF_HP_SURR_CLIP]), clip_hi = float(1.0 + a.hparams[PPOAF_HP_SURR_CLIP]);
    const float vf_clip = float(a.hparams[PPOAF_HP_VF_CLIP]);
    const bool gaussian = a.head == PPOAF_HEAD_GAUSSIAN_TANH;
    const int smp = tid / kG;                                        // sample slot inside the CTA

    // ---- every global load that does not depend on the cursor is issued first: the hidden activations of this
    // sample and the head weights travel while the cursor -> permutation -> dataset chain resolves ----
    const HeadSmem hs(a, s_dyn);
    // Everything up to pdl_wait() reads only data that no launch of the current step writes (parameters, the
    // dataset, the permutation, the cursor): it overlaps the tail of the previous launch.
    float4 ha[kFusedMaxChunks], hc[kFusedMaxChunks];
    float4 wreg[kFusedStageSlots];
    if constexpr (FUSED) {
        const int qa = a.Ha / 4;
#pragma unroll
        for (int k = 0; k < kFusedStageSlots; ++k) {                 // W_actor, coalesced 16-byte loads into registers
            const int t = tid + k * kLossThreads;
            const int row = t / qa, c4 = t - row * qa;
            wreg[k] = row < a.pred_dim ? *reinterpret_cast<const float4*>(a.W_actor + int64_t(row) * a.Ha + 4 * c4)
                                       : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    const int cur = *a.cursor;
    const int64_t* idx = a.perm + int64_t(cur) * a.batch_size;
    const int64_t j = live ? idx[i] : 0;
    const int64_t nxt = int64_t(cur + 1) * a.batch_size + i;
    const int64_t jn = (a.pf_rows[0] && live && nxt < a.n_flat) ? a.perm[nxt] : -1;
    float adv_mu = 0.f, adv_sd = 1.f, val_mu = 0.f, val_sd = 1.f;    // this minibatch's normalisation constants
    if (a.normalize_adv) { adv_mu = a.mb_adv_stats[2 * cur]; adv_sd = a.mb_adv_stats[2 * cur + 1]; }
    if (a.normalize_values) { val_mu = a.mb_val_stats[2 * cur]; val_sd = a.mb_val_stats[2 * cur + 1]; }

    if (gaussian && tid < a.act_dim) s_sd[tid] = std_of_log_std(a.log_std[tid], a.min_std, s_dsd[tid]);
    float adv = live ? a.advantages[j] : 0.f;
    const float lp_old = live ? a.log_probs[j] : 0.f;
    float target = live ? a.rewards_to_go[j] : 0.f;
    pdl_wait();
    pdl_trigger();
    if constexpr (FUSED) {
        const float* hra = a.h_actor + int64_t(live ? i : 0) * a.Ha + 4 * gl;
        const float* hrc = a.h_critic + int64_t(live ? i : 0) * a.Hc + 4 * gl;
#pragma unroll
        for (int c = 0; c < kFusedMaxChunks; ++c) {
            const int col = 4 * (gl + kG * c);
            ha[c] = (col < a.Ha && live) ? *reinterpret_cast<const float4*>(hra + 4 * kG * c) : make_float4(0.f, 0.f, 0.f, 0.f);
            hc[c] = (col < a.Hc && live) ? *reinterpret_cast<const float4*>(hrc + 4 * kG * c) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        const int qa = a.Ha / 4;
#pragma unroll
        for (int k = 0; k < kFusedStageSlots; ++k) {
            const int t = tid + k * kLossThreads;
            const int row = t / qa, c4 = t - row * qa;
            if (row < hs.prows) *reinterpret_cast<float4*>(hs.wa + row * hs.ldw + 4 * c4) = wreg[k];   // padding rows are zero
        }
        for (int t = tid; t < a.Hc / 4; t += kLossThreads)
            *reinterpret_cast<float4*>(hs.wc + 4 * t) = *reinterpret_cast<const float4*>(a.W_critic + 4 * t);
        if (tid < a.pred_dim) hs.b[tid] = a.b_actor[tid];
        if (tid == 0) hs.b[a.pred_dim] = a.b_critic[0];
    }
    if (jn >= 0) {
        // pull the NEXT minibatch's observation rows into L2 while this step's backward pass runs: the first-layer
        // GEMMs of the next step then gather from L2 instead of HBM
        const char* r0 = reinterpret_cast<const char*>(a.pf_rows[0]) + jn * a.pf_row_bytes[0];
        const char* r1 = reinterpret_cast<const char*>(a.pf_rows[1]) + jn * a.pf_row_bytes[1];
        for (int o = gl * 128; o < a.pf_row_bytes[0]; o += kG * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r0 + o));
        for (int o = gl * 128; o < a.pf_row_bytes[1]; o += kG * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r1 + o));
    }
    LOSS_STAMP(0);
    __syncthreads();
    LOSS_STAMP(1);

    float sc[kLossScalars];
#pragma unroll
    for (int k = 0; k < kLossScalars; ++k) sc[k] = 0.f;
    float dsd[kPerLane];                                             // d loss / d std for dims gl + 32k of this sample
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) dsd[k] = 0.f;

    if (a.normalize_adv) adv = (adv - adv_mu) / adv_sd;
    if (a.normalize_values) target = (target - val_mu) / val_sd;
    float v_fused = 0.f;
    if constexpr (FUSED) v_fused = head_forward(a, hs, ha, hc, gl, hs.pred + smp * kFusedPredLd);
    LOSS_STAMP(3);
    const float v = FUSED ? (live ? v_fused : 0.f) : (live ? a.critic_out[i] : 0.f);
    if (live && gl == 0) a.values[j] = v;                            // dataset.values[batch_idxs] = values (ppo.py:2340)
    float bad_value = isnan(v) ? 1.f : 0.f;

    const float* pred = FUSED ? hs.pred + smp * kFusedPredLd : a.actor_out + int64_t(live ? i : 0) * a.pred_dim;
    float* dpred = a.d_actor_out + int64_t(live ? i : 0) * a.pred_dim;
    float* sdp = hs.dpred + smp * kFusedPredLd;                      // FUSED: dL/d(actor out) kept for the head's dX
    actor_head_loss<FUSED>(a, a.head, live, gl, j, pred, dpred, sdp, s_sd, adv, lp_old, inv_b, w_ent, clip_lo, clip_hi,
                           sc, dsd, bad_value);

    LOSS_STAMP(4);
    // ---------------- critic ----------------
    float dv1 = 0.f;
    if (FUSED || (gl == 0 && live)) sc[LS_CRITIC] = critic_term(v, target, a.use_huber, dv1);
    if (FUSED && !(gl == 0 && live)) sc[LS_CRITIC] = 0.f;
    if (gl == 0 && live) {
        if (a.vf_clip_enabled) {
            const float vc = fminf(fmaxf(v, -vf_clip), vf_clip);
            float dv2;
            sc[LS_CRITIC_CLIPPED] = critic_term(vc, target, a.use_huber, dv2);
            const float pass = (v >= -vf_clip && v <= vf_clip) ? 1.f : 0.f;
            a.d_critic_out[i] = dv1 * inv_b;                                         // combined by vf_select_kernel
            a.d_critic_out[a.batch + i] = dv2 * pass * inv_b;
        } else {
            a.d_critic_out[i] = dv1 * inv_b;
        }
    }
    const float bad_any = group_max(bad_value);
    sc[LS_BAD_VALUE] = (live && gl == 0) ? bad_any : 0.f;

    if constexpr (FUSED) head_backward(a, hs, ha, hc, sdp, dv1, inv_b, live, gl, live ? i : 0);

    LOSS_STAMP(5);
    // ---------------- CTA partials; the last CTA to finish folds them ----------------
    const int n_vals = kLossScalars + (gaussian ? a.act_dim : 0);
    double* part = reinterpret_cast<double*>(a.partials);
    loss_cta_partials(sc, dsd, n_vals, s_red, part, CtaBarrier{});
    LOSS_STAMP(6);
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    LOSS_STAMP(7);
    if (!s_last) return;
    __threadfence();
    LOSS_STAMP(8);

    // ---------------- last CTA: totals -> d(log_std), epoch statistics, value-clip weights -----------
    loss_fold(a, n_vals, s_dsd, s_red, s_tot, s_sq, CtaBarrier{});
    if (tid == 0) {
        const double nb = double(a.batch);
        float critic_mean = float(s_tot[LS_CRITIC] / nb);
        if (a.vf_clip_enabled) {
            // critic_loss = max(loss(v), loss(clamp(v)))  (ppo.py:2427-2436; intended semantics, SURVEY Q4);
            // torch.max of two scalars splits the gradient evenly on a tie.
            const float clipped_mean = float(s_tot[LS_CRITIC_CLIPPED] / nb);
            float w1 = 1.f, w2 = 0.f;
            if (clipped_mean > critic_mean) { w1 = 0.f; w2 = 1.f; critic_mean = clipped_mean; }
            else if (clipped_mean == critic_mean) { w1 = 0.5f; w2 = 0.5f; }
            float* wsel = reinterpret_cast<float*>(part + size_t(gridDim.x) * kPartialStride);
            wsel[0] = w1; wsel[1] = w2;
        }
        add_epoch_stats(a, s_tot, critic_mean, w_ent);
        *a.ticket = 0u;  // ready for the next launch
    }
    LOSS_STAMP(10);
}

__global__ void vf_select_kernel(float* __restrict__ d_critic_out, int batch, const float* __restrict__ wsel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    d_critic_out[i] = wsel[0] * d_critic_out[i] + wsel[1] * d_critic_out[batch + i];
}

size_t loss_workspace_bytes(int max_batch, int /*act_dim*/) {
    const size_t blocks = size_t((max_batch + kSamplesPerBlock - 1) / kSamplesPerBlock);
    return align_up(blocks * kPartialStride * sizeof(double) + 16, 256);
}

int launch_ppo_loss(const LossArgs& a, cudaStream_t s) {
    PPOAF_CHECK_ARG(a.act_dim >= 1 && a.act_dim <= kMaxAct && a.pred_dim >= 1 && a.pred_dim <= kMaxAct,
                    "ppo loss: act_dim / prediction width must be in [1, %d]", kMaxAct);
    PPOAF_CHECK_ARG(a.batch >= 2, "ppo loss: minibatches of fewer than 2 rows are skipped by the caller");
    const int blocks = (a.batch + kSamplesPerBlock - 1) / kSamplesPerBlock;
    if (a.fused) {
        PPOAF_CHECK_ARG(loss_head_fusable(a.pred_dim, a.Ha, a.Hc, a.vf_clip_enabled), "ppo loss: head layers are not fusable");
        const size_t smem = sizeof(float) * size_t((a.pred_dim + kPB - 1) / kPB * kPB * (a.Ha + 4) + a.Hc + ((a.pred_dim + 1 + 3) & ~3) +
                                                   2 * kSamplesPerBlock * kFusedPredLd);
        launch_chain(ppo_loss_kernel<true>, dim3(blocks), dim3(kLossThreads), smem, s, a);
    } else {
        launch_chain(ppo_loss_kernel<false>, dim3(blocks), dim3(kLossThreads), 0, s, a);
    }
    PPOAF_CHECK_LAUNCH("ppo_loss_kernel");
    if (a.vf_clip_enabled) {
        const float* wsel = reinterpret_cast<const float*>(reinterpret_cast<const double*>(a.partials) +
                                                           size_t(blocks) * kPartialStride);
        vf_select_kernel<<<(a.batch + 255) / 256, 256, 0, s>>>(a.d_critic_out, a.batch, wsel);
        PPOAF_CHECK_LAUNCH("vf_select_kernel");
    }
    return 0;
}

}  // namespace ppoaf

#ifdef PPOAF_GEMM_TIMING
extern "C" int ppoaf_debug_loss_stamps(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, ppoaf::g_loss_stamps, sizeof(long long) * 16) == cudaSuccess ? 0 : 1;
}
#endif

// ---- stand-alone heads (PPOPolicy.evaluate's distribution half, policies/ppo_policy.py:939-950, and rollout-time
// sampling, :729-794): one thread per row.  The Categorical head runs the multi-categorical kernels with a table of one
// section. ----
namespace ppoaf {

__global__ void head_evaluate_kernel(const float* __restrict__ actor_out, int pred_dim, const float* __restrict__ log_std,
                                     float min_std, const float* __restrict__ actions, int act_dim, int n_rows,
                                     float* __restrict__ lp_out, float* __restrict__ ent_out) {
    __shared__ float s_sd[kMaxAct];
    float dstd;
    if (threadIdx.x < act_dim) s_sd[threadIdx.x] = std_of_log_std(log_std[threadIdx.x], min_std, dstd);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const float* x = actions + int64_t(i) * act_dim;
    float nsum = 0.f, slog = 0.f, ensum = 0.f, eslog = 0.f;
    for (int d = 0; d < act_dim; ++d) {
        const float mu = pred[d], sd = s_sd[d], z = x[d] - mu, lsd = logf(sd);
        nsum += fminf(fmaxf(-(z * z) / (2.f * (sd * sd)) - lsd - kLogSqrt2Pi, -100.f), 100.f);
        const float th = tanhf(x[d]);
        slog += logf(fmaxf(1.f - th * th, 1e-6f));
        ensum += fminf(fmaxf(-lsd - kLogSqrt2Pi, -100.f), 100.f);
        const float thm = tanhf(mu);
        eslog += logf(fmaxf(1.f - thm * thm, 1e-6f));
    }
    lp_out[i] = nsum - slog;
    if (ent_out) ent_out[i] = -(ensum - eslog);
}

// The random draws come from the HOST generator in the order the reference's CPU sampling consumes them (`noise`), so
// the actions are the reference's actions; everything else -- scaling by std, tanh squashing, range mapping, log-prob --
// happens here.  noise = N(0,1) [n, act_dim];  raw = noise * std + mean  (torch.normal: mul_ then add_);
// action = tanh(raw), mapped to [min, max] when given (distributions.py:560-610); log-prob :518-558
__global__ void head_sample_kernel(const float* __restrict__ actor_out, int pred_dim, const float* __restrict__ log_std,
                                   float min_std, const float* __restrict__ noise, const float* __restrict__ dist_min,
                                   const float* __restrict__ dist_max, int act_dim, int n_rows, float* __restrict__ raw_out,
                                   float* __restrict__ act_out, float* __restrict__ lp_out) {
    __shared__ float s_sd[kMaxAct];
    float dstd;
    if (threadIdx.x < act_dim) s_sd[threadIdx.x] = std_of_log_std(log_std[threadIdx.x], min_std, dstd);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const float* z = noise + int64_t(i) * act_dim;
    float* raw = raw_out + int64_t(i) * act_dim;
    float* act = act_out + int64_t(i) * act_dim;
    float nsum = 0.f, slog = 0.f;
    for (int d = 0; d < act_dim; ++d) {
        const float mu = pred[d], sd = s_sd[d];
        const float x = __fadd_rn(__fmul_rn(z[d], sd), mu);
        const float th = tanhf(x);
        float a = th;
        if (dist_min && dist_max)
            a = __fadd_rn(__fmul_rn(__fdiv_rn(__fadd_rn(th, 1.f), 2.f), __fsub_rn(dist_max[d], dist_min[d])), dist_min[d]);
        raw[d] = x;
        act[d] = a;
        const float dz = x - mu;
        nsum += fminf(fmaxf(-(dz * dz) / (2.f * (sd * sd)) - logf(sd) - kLogSqrt2Pi, -100.f), 100.f);
        slog += logf(fmaxf(1.f - th * th, 1e-6f));
    }
    lp_out[i] = nsum - slog;
}

// Multi-categorical evaluation; actions: int64 rows of act_ld (the number of sections; act_dim for the Categorical ABI)
__global__ void multi_categorical_evaluate_kernel(const float* __restrict__ actor_out, int pred_dim,
                                                  unsigned long long ends, const int64_t* __restrict__ actions,
                                                  int act_ld, int n_rows, float* __restrict__ lp_out,
                                                  float* __restrict__ ent_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const int64_t* act = actions + int64_t(i) * act_ld;
    float mx = pred[0];
    for (int c = 1; c < pred_dim; ++c) mx = fmaxf(mx, pred[c]);
    float se = 0.f;
    for (int c = 0; c < pred_dim; ++c) se += expf(pred[c] - mx);
    float lp = 0.f, h = 0.f;
    for (int o = 0, k = 0, c = 0; c < pred_dim; ++c) {
        if (!((ends >> c) & 1ull)) continue;
        float S = 0.f;                                            // section k = columns o .. c
        for (int d = o; d <= c; ++d) S += expf(pred[d] - mx) / se;
        const int a = int(act[k]);
        for (int d = o; d <= c; ++d) {
            const float pn = (expf(pred[d] - mx) / se) / S;
            const float l = logf(fminf(fmaxf(pn, kCatEps), 1.f - kCatEps));
            h += pn * l;
            if (d - o == a) lp += l;
        }
        o = c + 1;
        ++k;
    }
    lp_out[i] = lp;
    if (ent_out) ent_out[i] = -h;
}

// Multi-categorical sampling.  probs: the softmax of the whole row; noise: section k's Exp(1) block [n_rows, n_k] starts
// at n_rows * o_k; in each section a_k = first argmax(p~_k / q_k) (aten multinomial, one draw; distributions.py:223-249).
// raw_out (nullable): a second copy of the actions, which the Categorical ABI writes.  16 blocks of 128 per SM keep it
// at 32 registers, full occupancy.
__global__ void __launch_bounds__(128, 16)
multi_categorical_sample_kernel(const float* __restrict__ probs, int pred_dim, unsigned long long ends,
                                const float* __restrict__ noise, int n_sections, int n_rows, int64_t* __restrict__ act_out,
                                float* __restrict__ lp_out, int64_t* __restrict__ raw_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* p = probs + int64_t(i) * pred_dim;
    int64_t* act = act_out + int64_t(i) * n_sections;
    int64_t* raw = raw_out ? raw_out + int64_t(i) * n_sections : nullptr;
    float lp = 0.f;
    for (int o = 0, k = 0, c = 0; c < pred_dim; ++c) {
        if (!((ends >> c) & 1ull)) continue;
        const int nk = c - o + 1;
        const float* q = noise + int64_t(n_rows) * o + int64_t(i) * nk;
        float S = 0.f;
        for (int d = 0; d < nk; ++d) S += p[o + d];
        int best = 0;
        float best_v = -INFINITY, best_p = 0.f;
        for (int d = 0; d < nk; ++d) {
            const float pn = p[o + d] / S;
            const float v = pn / q[d];
            if (v > best_v) { best_v = v; best = d; best_p = pn; }        // first maximum, like argmax
        }
        act[k] = best;
        if (raw) raw[k] = best;
        lp += logf(fminf(fmaxf(best_p, kCatEps), 1.f - kCatEps));
        o = c + 1;
        ++k;
    }
    lp_out[i] = lp;
}

// Bernoulli (MultiBinary) evaluation: log-prob of fp32 0/1 actions [n_rows, k] and entropy, summed over the k columns,
// from the actor's logits [n_rows, k]
__global__ void bernoulli_evaluate_kernel(const float* __restrict__ actor_out, int k, const float* __restrict__ actions,
                                          int n_rows, float* __restrict__ lp_out, float* __restrict__ ent_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* z = actor_out + int64_t(i) * k;
    const float* x = actions + int64_t(i) * k;
    float lp = 0.f, h = 0.f;
    for (int c = 0; c < k; ++c) {
        const float p = sigmoid_f(z[c]), l = bernoulli_logit(p), ls = log_sigmoid(l);
        lp += ls - (1.f - x[c]) * l;
        h += (1.f - p) * l - ls;
    }
    lp_out[i] = lp;
    if (ent_out) ent_out[i] = h;
}

// Bernoulli sampling from the actor's logits [n_rows, k]: noise holds the host generator's U[0,1) draws [n_rows, k]
// (torch.rand, which Bernoulli(probs).sample() consumes the same way) and a = (u < sigmoid(z)) as fp32 0/1; all 0.5
// gives the deterministic action [p > 0.5].  Writes whichever of raw_out / act_out is given, and the summed log-prob.
__global__ void bernoulli_sample_kernel(const float* __restrict__ actor_out, int k, const float* __restrict__ noise,
                                        int n_rows, float* __restrict__ raw_out, float* __restrict__ act_out,
                                        float* __restrict__ lp_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* z = actor_out + int64_t(i) * k;
    const float* u = noise + int64_t(i) * k;
    float lp = 0.f;
    for (int c = 0; c < k; ++c) {
        const float p = sigmoid_f(z[c]), l = bernoulli_logit(p);
        const float x = u[c] < p ? 1.f : 0.f;
        if (raw_out) raw_out[int64_t(i) * k + c] = x;
        if (act_out) act_out[int64_t(i) * k + c] = x;
        lp += log_sigmoid(l) - (1.f - x) * l;
    }
    lp_out[i] = lp;
}

}  // namespace ppoaf

extern "C" int ppoaf_head_sample(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                                 float min_std, const float* noise, const float* dist_min, const float* dist_max,
                                 int32_t act_dim, int32_t n_rows, void* raw_action_out, void* action_out,
                                 float* log_prob_out, void* stream) {
    using namespace ppoaf;
    PPOAF_CHECK_ARG(head == PPOAF_HEAD_GAUSSIAN_TANH || head == PPOAF_HEAD_CATEGORICAL || head == PPOAF_HEAD_BERNOULLI,
                    "ppoaf_head_sample: unknown head");
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= kMaxAct && pred_dim >= 1 && pred_dim <= kMaxAct,
                    "ppoaf_head_sample: widths must be in [1, %d]", kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0 && noise != nullptr, "ppoaf_head_sample: bad arguments");
    PPOAF_CHECK_ARG((dist_min == nullptr) == (dist_max == nullptr), "ppoaf_head_sample: give both range bounds or neither");
    if (head == PPOAF_HEAD_BERNOULLI) {
        PPOAF_CHECK_ARG(pred_dim == act_dim, "ppoaf_head_sample: Bernoulli actor output width must equal act_dim");
        PPOAF_CHECK_ARG(log_std == nullptr && dist_min == nullptr,
                        "ppoaf_head_sample: the Bernoulli head takes no log_std and no range bounds");
    }
    if (n_rows == 0) return 0;
    const dim3 grid((n_rows + 127) / 128), block(128);
    if (head == PPOAF_HEAD_GAUSSIAN_TANH)
        head_sample_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, pred_dim, log_std, min_std, noise, dist_min, dist_max, act_dim, n_rows, static_cast<float*>(raw_action_out),
            static_cast<float*>(action_out), log_prob_out);
    else if (head == PPOAF_HEAD_BERNOULLI)
        bernoulli_sample_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, act_dim, noise, n_rows, static_cast<float*>(raw_action_out), static_cast<float*>(action_out),
            log_prob_out);
    else
        multi_categorical_sample_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, pred_dim, 1ull << (pred_dim - 1), noise, 1, n_rows, static_cast<int64_t*>(action_out), log_prob_out,
            static_cast<int64_t*>(raw_action_out));
    PPOAF_CHECK_LAUNCH("ppoaf_head_sample");
    return 0;
}

extern "C" int ppoaf_head_evaluate(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                                   float min_std, const void* actions, int32_t act_dim, int32_t n_rows,
                                   float* log_prob_out, float* entropy_out, void* stream) {
    using namespace ppoaf;
    PPOAF_CHECK_ARG(head == PPOAF_HEAD_GAUSSIAN_TANH || head == PPOAF_HEAD_CATEGORICAL || head == PPOAF_HEAD_BERNOULLI,
                    "ppoaf_head_evaluate: unknown head");
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= kMaxAct && pred_dim >= 1 && pred_dim <= kMaxAct,
                    "ppoaf_head_evaluate: widths must be in [1, %d]", kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_head_evaluate: n_rows < 0");
    if (head == PPOAF_HEAD_BERNOULLI) {
        PPOAF_CHECK_ARG(pred_dim == act_dim, "ppoaf_head_evaluate: Bernoulli actor output width must equal act_dim");
        PPOAF_CHECK_ARG(log_std == nullptr, "ppoaf_head_evaluate: the Bernoulli head takes no log_std");
    }
    if (n_rows == 0) return 0;
    const dim3 grid((n_rows + 127) / 128), block(128);
    if (head == PPOAF_HEAD_GAUSSIAN_TANH)
        head_evaluate_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, pred_dim, log_std, min_std, static_cast<const float*>(actions), act_dim, n_rows, log_prob_out, entropy_out);
    else if (head == PPOAF_HEAD_BERNOULLI)
        bernoulli_evaluate_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, act_dim, static_cast<const float*>(actions), n_rows, log_prob_out, entropy_out);
    else
        multi_categorical_evaluate_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
            actor_out, pred_dim, 1ull << (pred_dim - 1), static_cast<const int64_t*>(actions), act_dim, n_rows,
            log_prob_out, entropy_out);
    PPOAF_CHECK_LAUNCH("ppoaf_head_evaluate");
    return 0;
}

extern "C" int ppoaf_multi_categorical_evaluate(const float* actor_out, int32_t pred_dim, uint32_t section_ends_lo,
                                                uint32_t section_ends_hi, const int64_t* actions_i64, int32_t n_sections,
                                                int32_t n_rows, float* log_prob_out, float* entropy_out, void* stream) {
    using namespace ppoaf;
    const unsigned long long ends = (uint64_t(section_ends_hi) << 32) | section_ends_lo;
    PPOAF_CHECK_ARG(section_table_ok(ends, pred_dim, n_sections),
                    "ppoaf_multi_categorical_evaluate: bad section table for %d outputs / %d sections (at most %d outputs)",
                    pred_dim, n_sections, kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_multi_categorical_evaluate: n_rows < 0");
    if (n_rows == 0) return 0;
    multi_categorical_evaluate_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        actor_out, pred_dim, ends, actions_i64, n_sections, n_rows, log_prob_out, entropy_out);
    PPOAF_CHECK_LAUNCH("ppoaf_multi_categorical_evaluate");
    return 0;
}

extern "C" int ppoaf_multi_categorical_sample(const float* probs, int32_t pred_dim, uint32_t section_ends_lo,
                                              uint32_t section_ends_hi, const float* noise, int32_t n_sections,
                                              int32_t n_rows, int64_t* actions_out_i64, float* log_prob_out,
                                              void* stream) {
    using namespace ppoaf;
    const unsigned long long ends = (uint64_t(section_ends_hi) << 32) | section_ends_lo;
    PPOAF_CHECK_ARG(section_table_ok(ends, pred_dim, n_sections),
                    "ppoaf_multi_categorical_sample: bad section table for %d outputs / %d sections (at most %d outputs)",
                    pred_dim, n_sections, kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_multi_categorical_sample: n_rows < 0");
    if (n_rows == 0) return 0;
    PPOAF_CHECK_ARG(noise != nullptr, "ppoaf_multi_categorical_sample: noise is required");
    multi_categorical_sample_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        probs, pred_dim, ends, noise, n_sections, n_rows, actions_out_i64, log_prob_out, nullptr);
    PPOAF_CHECK_LAUNCH("ppoaf_multi_categorical_sample");
    return 0;
}
