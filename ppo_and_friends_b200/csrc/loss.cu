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

// d loss / d value of one live sample i (dv1: d critic_term(v) / dv) to d_critic_out; with value clipping also the
// clipped branch and its critic term, the two combined by vf_select_kernel
__device__ __forceinline__ void store_critic_grads(const LossArgs& a, int i, float v, float target, float dv1, float inv_b,
                                                   float vf_clip, float (&sc)[kLossScalars]) {
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

// Last CTA, one thread, from the totals: the value-clip branch weights (after the gridDim.x CTA partials of `stride`
// doubles), the epoch statistics, and the ticket reset for the next launch
__device__ __forceinline__ void loss_epilogue(const LossArgs& a, const double* s_tot, double* part, int stride, float w_ent) {
    const double nb = double(a.batch);
    float critic_mean = float(s_tot[LS_CRITIC] / nb);
    if (a.vf_clip_enabled) {
        // critic_loss = max(loss(v), loss(clamp(v)))  (ppo.py:2427-2436; intended semantics, SURVEY Q4);
        // torch.max of two scalars splits the gradient evenly on a tie.
        const float clipped_mean = float(s_tot[LS_CRITIC_CLIPPED] / nb);
        float w1 = 1.f, w2 = 0.f;
        if (clipped_mean > critic_mean) { w1 = 0.f; w2 = 1.f; critic_mean = clipped_mean; }
        else if (clipped_mean == critic_mean) { w1 = 0.5f; w2 = 0.5f; }
        float* wsel = reinterpret_cast<float*>(part + size_t(gridDim.x) * stride);
        wsel[0] = w1; wsel[1] = w2;
    }
    add_epoch_stats(a, s_tot, critic_mean, w_ent);
    *a.ticket = 0u;  // ready for the next launch
}

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
    if (gl == 0 && live) store_critic_grads(a, i, v, target, dv1, inv_b, vf_clip, sc);
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
    if (tid == 0) loss_epilogue(a, s_tot, part, kPartialStride, w_ent);
    LOSS_STAMP(10);
}

// ---- wide heads: Categorical rows of more than kMaxAct classes and Gaussian rows of more than kMaxAct dims ----
// One CTA per sample (wide_samples(head) samples per CTA, one after the other): the threads stride over the row, and
// every row-wide sum is a block reduction in a fixed order.  The row is re-read for each pass; after the first pass it
// comes from L1 / L2.  The actor's head layer is never fused here (kFusedMaxPred < kMaxAct).  The CTA partials hold
// kLossScalars sums and, for the Gaussian head, one fp64 sum of dL/d std per dimension (wide_partial_stride).
constexpr int kWideThreads = 256;
constexpr int kWideGaussianSamples = 8;     // the Gaussian head's per-dimension partials: fewer CTAs to fold
__host__ __device__ __forceinline__ int wide_samples(int head) { return head == PPOAF_HEAD_GAUSSIAN_TANH ? kWideGaussianSamples : 1; }
__host__ __device__ __forceinline__ int wide_partial_stride(int head, int act_dim) {
    return kLossScalars + (head == PPOAF_HEAD_GAUSSIAN_TANH ? act_dim : 0);
}

// Block-wide sums (or maxima) of N values at once; the result is in every thread.  scratch: 32 N floats.
template <int N, bool MAX>
__device__ __forceinline__ void block_reduce_n(float (&v)[N], float* scratch) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < N; ++k)
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float y = __shfl_xor_sync(kFull, v[k], o);
            v[k] = MAX ? fmaxf(v[k], y) : v[k] + y;
        }
    __syncthreads();                                                 // the previous reduction has read scratch
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < N; ++k) scratch[k * 32 + warp] = v[k];
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < N; ++k) {
        v[k] = lane < kWideThreads / 32 ? scratch[k * 32 + lane] : (MAX ? -INFINITY : 0.f);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float y = __shfl_xor_sync(kFull, v[k], o);
            v[k] = MAX ? fmaxf(v[k], y) : v[k] + y;
        }
    }
}

// One column of the Categorical head: p = softmax(z)_c, pn = p / S (Categorical(probs) renormalises), lg = log of pn
// clamped to [eps, 1 - eps]
struct CatColumn { float p, pn, lg; };
__device__ __forceinline__ CatColumn cat_column(float z, float mx, float se, float S) {
    CatColumn r;
    r.p = expf(z - mx) / se;
    r.pn = r.p / S;
    r.lg = logf(fminf(fmaxf(r.pn, kCatEps), 1.f - kCatEps));
    return r;
}

// The Categorical branch of actor_head_loss on a row of n = pred_dim logits with one section: writes dL/dz to dpred and
// the sample's scalars to sc (thread 0); returns 1 when a logit is NaN
__device__ __forceinline__ float wide_categorical_loss(const LossArgs& a, const float* pred, float* dpred, int64_t act,
                                                      float adv, float lp_old, float inv_b, float w_ent, float clip_lo,
                                                      float clip_hi, float (&sc)[kLossScalars], float* red) {
    const int n = a.pred_dim, tid = threadIdx.x;
    float mb[2] = {-INFINITY, 0.f};                                  // max logit, NaN seen
    for (int c = tid; c < n; c += kWideThreads) {
        const float z = pred[c];
        mb[0] = fmaxf(mb[0], z);
        mb[1] = fmaxf(mb[1], isnan(z) ? 1.f : 0.f);
    }
    block_reduce_n<2, true>(mb, red);
    const float mx = mb[0];
    float se[1] = {0.f};
    for (int c = tid; c < n; c += kWideThreads) se[0] += expf(pred[c] - mx);
    block_reduce_n<1, false>(se, red);
    float S[1] = {0.f};
    for (int c = tid; c < n; c += kWideThreads) S[0] += expf(pred[c] - mx) / se[0];
    block_reduce_n<1, false>(S, red);
    float h[1] = {0.f};
    for (int c = tid; c < n; c += kWideThreads) {
        const CatColumn k = cat_column(pred[c], mx, se[0], S[0]);
        h[0] += k.pn * k.lg;
    }
    block_reduce_n<1, false>(h, red);
    const bool hit_any = act >= 0 && act < n;
    const float lp = hit_any ? cat_column(pred[act], mx, se[0], S[0]).lg : 0.f;
    const float g_lp = ppo_surrogate(lp, -h[0], lp_old, adv, inv_b, clip_lo, clip_hi, tid == 0, sc);
    const float g_ent = -w_ent * inv_b;                               // dL/dH_i
    // G_c = dL/d pn_c ; pn = p / S ; p = softmax(z)
    auto G_of = [&](int c, const CatColumn& k) {
        const float q = fminf(fmaxf(k.pn, kCatEps), 1.f - kCatEps);
        const float mask = (k.pn >= kCatEps && k.pn <= 1.f - kCatEps) ? 1.f : 0.f;
        const float dlg = (c == act ? g_lp : 0.f) + g_ent * (-k.pn);
        return g_ent * (-k.lg) + dlg * mask / q;
    };
    float gdotp[1] = {0.f};
    for (int c = tid; c < n; c += kWideThreads) {
        const CatColumn k = cat_column(pred[c], mx, se[0], S[0]);
        gdotp[0] += G_of(c, k) * k.p;
    }
    block_reduce_n<1, false>(gdotp, red);
    const float s = S[0], gp = gdotp[0];
    float dpdotp[1] = {0.f};
    for (int c = tid; c < n; c += kWideThreads) {
        const CatColumn k = cat_column(pred[c], mx, se[0], s);
        dpdotp[0] += (G_of(c, k) / s - gp / (s * s)) * k.p;          // dL/dp_c p_c
    }
    block_reduce_n<1, false>(dpdotp, red);
    for (int c = tid; c < n; c += kWideThreads) {
        const CatColumn k = cat_column(pred[c], mx, se[0], s);
        dpred[c] = k.p * ((G_of(c, k) / s - gp / (s * s)) - dpdotp[0]);
    }
    return mb[1];
}

// The Gaussian-tanh branch of actor_head_loss on a row of act_dim means: writes dL/d mu to dpred, adds dL/d std of every
// dimension to acc (the thread that owns it) and the sample's scalars to sc (thread 0); returns 1 when a mean is NaN
__device__ __forceinline__ float wide_gaussian_loss(const LossArgs& a, const float* pred, float* dpred, const float* x,
                                                   float adv, float lp_old, float inv_b, float w_ent, float clip_lo,
                                                   float clip_hi, float (&sc)[kLossScalars], double* acc, float* red) {
    const int n = a.act_dim, tid = threadIdx.x;
    float s5[5] = {0.f, 0.f, 0.f, 0.f, 0.f};                         // nsum, slog, ensum, eslog, NaN means
    for (int d = tid; d < n; d += kWideThreads) {
        float dstd;
        const float sd = std_of_log_std(a.log_std[d], a.min_std, dstd), mu = pred[d], xd = x[d], z = xd - mu;
        s5[4] += isnan(mu) ? 1.f : 0.f;
        const float lsd = logf(sd);
        s5[0] += fminf(fmaxf(-(z * z) / (2.f * (sd * sd)) - lsd - kLogSqrt2Pi, -100.f), 100.f);   // Normal.log_prob
        const float th = tanhf(xd);
        s5[1] += logf(fmaxf(1.f - th * th, 1e-6f));
        s5[2] += fminf(fmaxf(-lsd - kLogSqrt2Pi, -100.f), 100.f);                               // log N(mu; mu, sd)
        const float thm = tanhf(mu);
        s5[3] += logf(fmaxf(1.f - thm * thm, 1e-6f));
    }
    block_reduce_n<5, false>(s5, red);
    const float lp = s5[0] - s5[1];
    const float ent = -(s5[2] - s5[3]);                                // entropy = -log_prob(mean) (:694)
    const float g_lp = ppo_surrogate(lp, ent, lp_old, adv, inv_b, clip_lo, clip_hi, tid == 0, sc);
    const float g_ent = -w_ent * inv_b;
    for (int d = tid; d < n; d += kWideThreads) {
        float dstd;
        const float sd = std_of_log_std(a.log_std[d], a.min_std, dstd), mu = pred[d], z = x[d] - mu, var = sd * sd;
        const float lsd = logf(sd);
        const float nl = -(z * z) / (2.f * var) - lsd - kLogSqrt2Pi, nle = -lsd - kLogSqrt2Pi;
        const float on = (nl >= -100.f && nl <= 100.f) ? 1.f : 0.f, one = (nle >= -100.f && nle <= 100.f) ? 1.f : 0.f;
        const float thm = tanhf(mu);
        const float tmask = (1.f - thm * thm >= 1e-6f) ? 1.f : 0.f;
        // dlp/dmu = z/var ; dH/dmu = -2 tanh(mu) ; dlp/dsd = z^2/sd^3 - 1/sd ; dH/dsd = 1/sd
        dpred[d] = g_lp * on * (z / var) + g_ent * tmask * (-2.f * thm);
        acc[d] += double(g_lp * on * ((z * z) / (var * sd) - 1.f / sd) + g_ent * one * (1.f / sd));
    }
    return s5[4] > 0.f ? 1.f : 0.f;
}

__global__ void __launch_bounds__(kWideThreads) ppo_loss_wide_kernel(const LossArgs a) {
    extern __shared__ double s_acc[];                                // Gaussian: this CTA's sums of dL/d std [act_dim]
    __shared__ float s_red[5 * 32];
    __shared__ double s_sq[32];
    __shared__ double s_tot[kLossScalars];
    __shared__ bool s_last;

    const int tid = threadIdx.x;
    const float inv_b = 1.0f / float(a.batch);
    const float w_ent = float(a.hparams[PPOAF_HP_ENTROPY_WEIGHT]);
    const float clip_lo = float(1.0 - a.hparams[PPOAF_HP_SURR_CLIP]), clip_hi = float(1.0 + a.hparams[PPOAF_HP_SURR_CLIP]);
    const float vf_clip = float(a.hparams[PPOAF_HP_VF_CLIP]);
    const bool gaussian = a.head == PPOAF_HEAD_GAUSSIAN_TANH;
    const int spc = wide_samples(a.head), stride = wide_partial_stride(a.head, a.act_dim);
    // up to pdl_wait(): only data that no launch of the current step writes (as in ppo_loss_kernel)
    const int cur = *a.cursor;
    const int64_t* idx = a.perm + int64_t(cur) * a.batch_size;
    float adv_mu = 0.f, adv_sd = 1.f, val_mu = 0.f, val_sd = 1.f;
    if (a.normalize_adv) { adv_mu = a.mb_adv_stats[2 * cur]; adv_sd = a.mb_adv_stats[2 * cur + 1]; }
    if (a.normalize_values) { val_mu = a.mb_val_stats[2 * cur]; val_sd = a.mb_val_stats[2 * cur + 1]; }
    if (gaussian)
        for (int d = tid; d < a.act_dim; d += kWideThreads) s_acc[d] = 0.0;
    pdl_wait();
    pdl_trigger();

    double tot[kLossScalars];                                        // thread 0: this CTA's sums of the sample scalars
#pragma unroll
    for (int k = 0; k < kLossScalars; ++k) tot[k] = 0.0;
    for (int s = 0; s < spc; ++s) {
        const int i = blockIdx.x * spc + s;
        if (i >= a.batch) break;                                     // uniform over the CTA
        const int64_t j = idx[i];
        const int64_t nxt = int64_t(cur + 1) * a.batch_size + i;
        if (a.pf_rows[0] && nxt < a.n_flat) {                        // the next minibatch's rows into L2 (ppo_loss_kernel)
            const int64_t jn = a.perm[nxt];
            const char* r0 = reinterpret_cast<const char*>(a.pf_rows[0]) + jn * a.pf_row_bytes[0];
            const char* r1 = reinterpret_cast<const char*>(a.pf_rows[1]) + jn * a.pf_row_bytes[1];
            for (int o = tid * 128; o < a.pf_row_bytes[0]; o += kWideThreads * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r0 + o));
            for (int o = tid * 128; o < a.pf_row_bytes[1]; o += kWideThreads * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r1 + o));
        }
        float adv = a.advantages[j], target = a.rewards_to_go[j];
        const float lp_old = a.log_probs[j];
        if (a.normalize_adv) adv = (adv - adv_mu) / adv_sd;
        if (a.normalize_values) target = (target - val_mu) / val_sd;
        const float v = a.critic_out[i];
        float sc[kLossScalars];
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) sc[k] = 0.f;
        const float* pred = a.actor_out + int64_t(i) * a.pred_dim;
        float* dpred = a.d_actor_out + int64_t(i) * a.pred_dim;
        const float bad = gaussian
            ? wide_gaussian_loss(a, pred, dpred, reinterpret_cast<const float*>(a.raw_actions) + j * a.act_dim, adv,
                                 lp_old, inv_b, w_ent, clip_lo, clip_hi, sc, s_acc, s_red)
            : wide_categorical_loss(a, pred, dpred, reinterpret_cast<const int64_t*>(a.raw_actions)[j], adv, lp_old,
                                    inv_b, w_ent, clip_lo, clip_hi, sc, s_red);
        if (tid == 0) {
            a.values[j] = v;                                         // dataset.values[batch_idxs] = values (ppo.py:2340)
            float dv1;
            sc[LS_CRITIC] = critic_term(v, target, a.use_huber, dv1);
            store_critic_grads(a, i, v, target, dv1, inv_b, vf_clip, sc);
            sc[LS_BAD_VALUE] = fmaxf(bad, isnan(v) ? 1.f : 0.f);
#pragma unroll
            for (int k = 0; k < kLossScalars; ++k) tot[k] += double(sc[k]);
        }
    }

    // ---- CTA partials; the last CTA to finish folds them in CTA order ----
    double* part = reinterpret_cast<double*>(a.partials);
    if (tid == 0) {
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) part[size_t(blockIdx.x) * stride + k] = tot[k];
    }
    if (gaussian)
        for (int d = tid; d < a.act_dim; d += kWideThreads) part[size_t(blockIdx.x) * stride + kLossScalars + d] = s_acc[d];
    __threadfence();
    __syncthreads();
    if (tid == 0) s_last = atomicAdd(a.ticket, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!s_last) return;
    __threadfence();

    double my_sq = 0.0;
    for (int vi = tid; vi < stride; vi += kWideThreads) {
        double t = 0.0;
        for (unsigned b = 0; b < gridDim.x; ++b) t += __ldcg(&part[size_t(b) * stride + vi]);
        if (vi < kLossScalars) {
            s_tot[vi] = t;
        } else {
            float dstd;
            std_of_log_std(a.log_std[vi - kLossScalars], a.min_std, dstd);
            const float gls = float(t) * dstd;
            store_d_log_std(a, vi - kLossScalars, gls);
            my_sq += double(gls) * double(gls);
        }
    }
    my_sq = block_sum(my_sq, s_sq);                                  // its barriers also publish s_tot
    if (tid == 0) {
        if (a.sq_log_std) *a.sq_log_std = my_sq;
        loss_epilogue(a, s_tot, part, stride, w_ent);
    }
}

__global__ void vf_select_kernel(float* __restrict__ d_critic_out, int batch, const float* __restrict__ wsel) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= batch) return;
    d_critic_out[i] = wsel[0] * d_critic_out[i] + wsel[1] * d_critic_out[batch + i];
}

// CTA partials of the widest plan a configuration can launch, then the two value-clip weights.  act_dim > kMaxAct: the
// wide Gaussian head; the wide Categorical head (act_dim = 1, one CTA per sample) always fits the narrow kernel's size.
size_t loss_workspace_bytes(int max_batch, int act_dim) {
    const size_t blocks = size_t((max_batch + kSamplesPerBlock - 1) / kSamplesPerBlock);
    size_t doubles = blocks * kPartialStride;
    const size_t wide_cat = size_t(max_batch) * wide_partial_stride(PPOAF_HEAD_CATEGORICAL, 1);
    doubles = wide_cat > doubles ? wide_cat : doubles;
    if (act_dim > kMaxAct) {
        const size_t wide_gauss = size_t((max_batch + kWideGaussianSamples - 1) / kWideGaussianSamples) *
                                  wide_partial_stride(PPOAF_HEAD_GAUSSIAN_TANH, act_dim);
        doubles = wide_gauss > doubles ? wide_gauss : doubles;
    }
    return align_up(doubles * sizeof(double) + 16, 256);
}

// Rows of up to kMaxAct outputs run ppo_loss_kernel, wider Categorical / Gaussian rows ppo_loss_wide_kernel (whose
// head layers are never fused)
int launch_ppo_loss(const LossArgs& a, cudaStream_t s) {
    const bool wide = a.pred_dim > kMaxAct || a.act_dim > kMaxAct;
    if (wide)
        PPOAF_CHECK_ARG((a.head == PPOAF_HEAD_CATEGORICAL && a.act_dim == 1 && a.pred_dim <= kMaxCategoricalClasses) ||
                        (a.head == PPOAF_HEAD_GAUSSIAN_TANH && a.act_dim == a.pred_dim && a.pred_dim <= kMaxGaussianDims),
                        "ppo loss: head width %d is outside the bounds of head %d (Categorical <= %d, Gaussian <= %d, "
                        "others <= %d)", a.pred_dim, a.head, kMaxCategoricalClasses, kMaxGaussianDims, kMaxAct);
    else
        PPOAF_CHECK_ARG(a.act_dim >= 1 && a.pred_dim >= 1, "ppo loss: act_dim / prediction width must be >= 1");
    PPOAF_CHECK_ARG(a.batch >= 2, "ppo loss: minibatches of fewer than 2 rows are skipped by the caller");
    size_t wsel_at;                                                  // value-clip weights, in doubles past a.partials
    if (wide) {
        PPOAF_CHECK_ARG(!a.fused, "ppo loss: head layers of more than %d outputs are not fusable", kFusedMaxPred);
        const int spc = wide_samples(a.head), blocks = (a.batch + spc - 1) / spc;
        const size_t smem = a.head == PPOAF_HEAD_GAUSSIAN_TANH ? size_t(a.act_dim) * sizeof(double) : 0;
        launch_chain(ppo_loss_wide_kernel, dim3(blocks), dim3(kWideThreads), smem, s, a);
        PPOAF_CHECK_LAUNCH("ppo_loss_wide_kernel");
        wsel_at = size_t(blocks) * wide_partial_stride(a.head, a.act_dim);
    } else {
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
        wsel_at = size_t(blocks) * kPartialStride;
    }
    if (a.vf_clip_enabled) {
        const float* wsel = reinterpret_cast<const float*>(reinterpret_cast<const double*>(a.partials) + wsel_at);
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

// ---- wide stand-alone heads (rows of more than kMaxAct outputs): one warp per row, the lanes striding over it, with
// the per-element arithmetic of the one-thread-per-row kernels above ----
constexpr int kWideRowThreads = 256;
constexpr int kWideRowsPerCta = kWideRowThreads / 32;

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// s_sd: std of every dimension, computed once per CTA (dynamic shared memory, act_dim floats)
__device__ __forceinline__ void stage_std(const float* log_std, float min_std, int act_dim, float* s_sd) {
    float dstd;
    for (int d = threadIdx.x; d < act_dim; d += kWideRowThreads) s_sd[d] = std_of_log_std(log_std[d], min_std, dstd);
    __syncthreads();
}

__global__ void __launch_bounds__(kWideRowThreads)
gaussian_evaluate_wide_kernel(const float* __restrict__ actor_out, int pred_dim, const float* __restrict__ log_std,
                              float min_std, const float* __restrict__ actions, int act_dim, int n_rows,
                              float* __restrict__ lp_out, float* __restrict__ ent_out) {
    extern __shared__ float s_sd[];
    stage_std(log_std, min_std, act_dim, s_sd);
    const int lane = threadIdx.x & 31, i = blockIdx.x * kWideRowsPerCta + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const float* x = actions + int64_t(i) * act_dim;
    float nsum = 0.f, slog = 0.f, ensum = 0.f, eslog = 0.f;
    for (int d = lane; d < act_dim; d += 32) {
        const float mu = pred[d], sd = s_sd[d], z = x[d] - mu, lsd = logf(sd);
        nsum += fminf(fmaxf(-(z * z) / (2.f * (sd * sd)) - lsd - kLogSqrt2Pi, -100.f), 100.f);
        const float th = tanhf(x[d]);
        slog += logf(fmaxf(1.f - th * th, 1e-6f));
        ensum += fminf(fmaxf(-lsd - kLogSqrt2Pi, -100.f), 100.f);
        const float thm = tanhf(mu);
        eslog += logf(fmaxf(1.f - thm * thm, 1e-6f));
    }
    nsum = warp_sum(nsum); slog = warp_sum(slog); ensum = warp_sum(ensum); eslog = warp_sum(eslog);
    if (lane == 0) {
        lp_out[i] = nsum - slog;
        if (ent_out) ent_out[i] = -(ensum - eslog);
    }
}

__global__ void __launch_bounds__(kWideRowThreads)
gaussian_sample_wide_kernel(const float* __restrict__ actor_out, int pred_dim, const float* __restrict__ log_std,
                            float min_std, const float* __restrict__ noise, const float* __restrict__ dist_min,
                            const float* __restrict__ dist_max, int act_dim, int n_rows, float* __restrict__ raw_out,
                            float* __restrict__ act_out, float* __restrict__ lp_out) {
    extern __shared__ float s_sd[];
    stage_std(log_std, min_std, act_dim, s_sd);
    const int lane = threadIdx.x & 31, i = blockIdx.x * kWideRowsPerCta + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const float* z = noise + int64_t(i) * act_dim;
    float* raw = raw_out + int64_t(i) * act_dim;
    float* act = act_out + int64_t(i) * act_dim;
    float nsum = 0.f, slog = 0.f;
    for (int d = lane; d < act_dim; d += 32) {
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
    nsum = warp_sum(nsum); slog = warp_sum(slog);
    if (lane == 0) lp_out[i] = nsum - slog;
}

// Categorical evaluation on logits: softmax, Categorical(probs) (renormalise by S, clamp, log), entropy and the log-prob
// of the int64 index in column 0 of each actions row (act_ld int64 per row)
__global__ void __launch_bounds__(kWideRowThreads)
categorical_evaluate_wide_kernel(const float* __restrict__ actor_out, int pred_dim, const int64_t* __restrict__ actions,
                                 int act_ld, int n_rows, float* __restrict__ lp_out, float* __restrict__ ent_out) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * kWideRowsPerCta + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    float mx = -INFINITY;
    for (int c = lane; c < pred_dim; c += 32) mx = fmaxf(mx, pred[c]);
    mx = warp_max(mx);
    float se = 0.f;
    for (int c = lane; c < pred_dim; c += 32) se += expf(pred[c] - mx);
    se = warp_sum(se);
    float S = 0.f;
    for (int c = lane; c < pred_dim; c += 32) S += expf(pred[c] - mx) / se;
    S = warp_sum(S);
    float h = 0.f;
    for (int c = lane; c < pred_dim; c += 32) {
        const CatColumn k = cat_column(pred[c], mx, se, S);
        h += k.pn * k.lg;
    }
    h = warp_sum(h);
    if (lane == 0) {
        const int64_t a = actions[int64_t(i) * act_ld];
        lp_out[i] = (a >= 0 && a < pred_dim) ? cat_column(pred[a], mx, se, S).lg : 0.f;
        if (ent_out) ent_out[i] = -h;
    }
}

// Categorical sampling from softmax probs and Exp(1) noise [n_rows, pred_dim]: a = first argmax(p~ / q), p~ = p / S
// (the multi-categorical kernel's draw with one section); writes act_out and raw_out (nullable) and the log-prob
__global__ void __launch_bounds__(kWideRowThreads)
categorical_sample_wide_kernel(const float* __restrict__ probs, int pred_dim, const float* __restrict__ noise, int n_rows,
                               int64_t* __restrict__ act_out, float* __restrict__ lp_out, int64_t* __restrict__ raw_out) {
    const int lane = threadIdx.x & 31, i = blockIdx.x * kWideRowsPerCta + (threadIdx.x >> 5);
    if (i >= n_rows) return;
    const float* p = probs + int64_t(i) * pred_dim;
    const float* q = noise + int64_t(i) * pred_dim;
    float S = 0.f;
    for (int c = lane; c < pred_dim; c += 32) S += p[c];
    S = warp_sum(S);
    int best = pred_dim;                                              // past the row: loses every comparison
    float best_v = -INFINITY, best_p = 0.f;
    for (int c = lane; c < pred_dim; c += 32) {
        const float pn = p[c] / S;
        const float v = pn / q[c];
        if (v > best_v) { best_v = v; best = c; best_p = pn; }        // a lane's columns rise: its first maximum
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {                                // the first maximum of the row, like argmax
        const float ov = __shfl_xor_sync(kFull, best_v, o), op = __shfl_xor_sync(kFull, best_p, o);
        const int oc = __shfl_xor_sync(kFull, best, o);
        if (ov > best_v || (ov == best_v && oc < best)) { best_v = ov; best = oc; best_p = op; }
    }
    if (lane == 0) {
        if (best == pred_dim) best = 0;                               // no comparison held (NaN row): column 0
        act_out[i] = best;
        if (raw_out) raw_out[i] = best;
        lp_out[i] = logf(fminf(fmaxf(best_p, kCatEps), 1.f - kCatEps));
    }
}

// Widest rows a stand-alone head accepts (actor outputs and action columns alike), and which rows take the wide kernels
static int head_max_width(int head) {
    return head == PPOAF_HEAD_GAUSSIAN_TANH ? kMaxGaussianDims : head == PPOAF_HEAD_CATEGORICAL ? kMaxCategoricalClasses : kMaxAct;
}
static bool head_is_wide(int head, int pred_dim, int act_dim) {
    return head == PPOAF_HEAD_GAUSSIAN_TANH ? act_dim > kMaxAct : head == PPOAF_HEAD_CATEGORICAL && pred_dim > kMaxAct;
}

}  // namespace ppoaf

extern "C" int ppoaf_head_sample(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                                 float min_std, const float* noise, const float* dist_min, const float* dist_max,
                                 int32_t act_dim, int32_t n_rows, void* raw_action_out, void* action_out,
                                 float* log_prob_out, void* stream) {
    using namespace ppoaf;
    PPOAF_CHECK_ARG(head == PPOAF_HEAD_GAUSSIAN_TANH || head == PPOAF_HEAD_CATEGORICAL || head == PPOAF_HEAD_BERNOULLI,
                    "ppoaf_head_sample: unknown head");
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= head_max_width(head) && pred_dim >= 1 && pred_dim <= head_max_width(head),
                    "ppoaf_head_sample: head width %d / %d is outside 1 .. %d for head %d", pred_dim, act_dim,
                    head_max_width(head), head);
    PPOAF_CHECK_ARG(n_rows >= 0 && noise != nullptr, "ppoaf_head_sample: bad arguments");
    PPOAF_CHECK_ARG((dist_min == nullptr) == (dist_max == nullptr), "ppoaf_head_sample: give both range bounds or neither");
    if (head == PPOAF_HEAD_BERNOULLI) {
        PPOAF_CHECK_ARG(pred_dim == act_dim, "ppoaf_head_sample: Bernoulli actor output width must equal act_dim");
        PPOAF_CHECK_ARG(log_std == nullptr && dist_min == nullptr,
                        "ppoaf_head_sample: the Bernoulli head takes no log_std and no range bounds");
    }
    if (n_rows == 0) return 0;
    if (head_is_wide(head, pred_dim, act_dim)) {
        const dim3 grid((n_rows + kWideRowsPerCta - 1) / kWideRowsPerCta), block(kWideRowThreads);
        if (head == PPOAF_HEAD_GAUSSIAN_TANH)
            gaussian_sample_wide_kernel<<<grid, block, size_t(act_dim) * sizeof(float), (cudaStream_t)stream>>>(
                actor_out, pred_dim, log_std, min_std, noise, dist_min, dist_max, act_dim, n_rows,
                static_cast<float*>(raw_action_out), static_cast<float*>(action_out), log_prob_out);
        else
            categorical_sample_wide_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
                actor_out, pred_dim, noise, n_rows, static_cast<int64_t*>(action_out), log_prob_out,
                static_cast<int64_t*>(raw_action_out));
        PPOAF_CHECK_LAUNCH("ppoaf_head_sample(wide)");
        return 0;
    }
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
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= head_max_width(head) && pred_dim >= 1 && pred_dim <= head_max_width(head),
                    "ppoaf_head_evaluate: head width %d / %d is outside 1 .. %d for head %d", pred_dim, act_dim,
                    head_max_width(head), head);
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_head_evaluate: n_rows < 0");
    if (head == PPOAF_HEAD_BERNOULLI) {
        PPOAF_CHECK_ARG(pred_dim == act_dim, "ppoaf_head_evaluate: Bernoulli actor output width must equal act_dim");
        PPOAF_CHECK_ARG(log_std == nullptr, "ppoaf_head_evaluate: the Bernoulli head takes no log_std");
    }
    if (n_rows == 0) return 0;
    if (head_is_wide(head, pred_dim, act_dim)) {
        const dim3 grid((n_rows + kWideRowsPerCta - 1) / kWideRowsPerCta), block(kWideRowThreads);
        if (head == PPOAF_HEAD_GAUSSIAN_TANH)
            gaussian_evaluate_wide_kernel<<<grid, block, size_t(act_dim) * sizeof(float), (cudaStream_t)stream>>>(
                actor_out, pred_dim, log_std, min_std, static_cast<const float*>(actions), act_dim, n_rows, log_prob_out,
                entropy_out);
        else
            categorical_evaluate_wide_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(
                actor_out, pred_dim, static_cast<const int64_t*>(actions), act_dim, n_rows, log_prob_out, entropy_out);
        PPOAF_CHECK_LAUNCH("ppoaf_head_evaluate(wide)");
        return 0;
    }
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
