// Fused PPO loss, forward + backward, for one minibatch (reference ppo.py:2299-2438 with the
// distribution arithmetic of networks/distributions.py:491-558,694 and torch's Normal/Categorical).
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

template <bool FUSED>
__global__ void __launch_bounds__(kLossThreads) ppo_loss_kernel(const LossArgs a) {
    extern __shared__ __align__(16) float s_dyn[];      // FUSED: W_actor [pred][Ha+4] | W_critic [Hc] | biases | pred | dpred
    __shared__ float s_sd[kMaxAct], s_dsd[kMaxAct];
    __shared__ double s_red[kLossThreads / 32][kPartialStride];
    __shared__ double s_tot[kPartialStride];
    __shared__ bool s_last;

#ifdef PPOAF_GEMM_TIMING
    const long long t_entry = clock64();
#endif
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
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
    const int prows = (a.pred_dim + kPB - 1) / kPB * kPB;            // head rows padded to whole blocks of kPB
    const int ldw = a.Ha + 4;                                        // rows of W_actor land on distinct bank groups
    float* s_wa = s_dyn;                                             // [prows][ldw]
    float* s_wc = s_wa + prows * ldw;                                // [Hc]
    float* s_b = s_wc + a.Hc;                                        // [pred + 1]
    float* s_pred = s_b + ((a.pred_dim + 1 + 3) & ~3);               // [samples per block][kFusedPredLd]
    float* s_dpred = s_pred + kSamplesPerBlock * kFusedPredLd;
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

    if (gaussian && tid < a.act_dim) {
        // std = max(softplus(log_std), min_std)  (distributions.py:514-515) and d std / d log_std
        const float ls = a.log_std[tid];
        const float sp = softplus_torch(ls);
        s_sd[tid] = fmaxf(sp, a.min_std);
        const float sig = ls > 20.f ? 1.f : 1.f / (1.f + expf(-ls));
        s_dsd[tid] = sp > a.min_std ? sig : (sp == a.min_std ? 0.5f * sig : 0.f);
    }
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
            if (row < prows) *reinterpret_cast<float4*>(s_wa + row * ldw + 4 * c4) = wreg[k];   // padding rows are zero
        }
        for (int t = tid; t < a.Hc / 4; t += kLossThreads)
            *reinterpret_cast<float4*>(s_wc + 4 * t) = *reinterpret_cast<const float4*>(a.W_critic + 4 * t);
        if (tid < a.pred_dim) s_b[tid] = a.b_actor[tid];
        if (tid == 0) s_b[a.pred_dim] = a.b_critic[0];
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
    float dsd[kPerLane];                                             // d loss / d std for dims gl + 8k of this sample
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) dsd[k] = 0.f;

    if (a.normalize_adv) adv = (adv - adv_mu) / adv_sd;
    if (a.normalize_values) target = (target - val_mu) / val_sd;
    // ---- fused heads, forward: every lane dots its columns of the hidden activations with all head rows, the 8
    // lanes of the sample fold their partial sums, and the outputs go to shared memory ----
    float v_fused = 0.f;
    if constexpr (FUSED) {
        float acc[kFusedMaxPred];
#pragma unroll
        for (int d = 0; d < kFusedMaxPred; ++d) acc[d] = 0.f;
#pragma unroll
        for (int c = 0; c < kFusedMaxChunks; ++c) {
            const int col = 4 * (gl + kG * c);
            if (col < a.Ha) {
#pragma unroll
                for (int db = 0; db < kFusedMaxPred / kPB; ++db) {
                    if (db * kPB < a.pred_dim) {                     // uniform: whole blocks of independent rows
                        float4 w[kPB];
#pragma unroll
                        for (int e = 0; e < kPB; ++e) w[e] = *reinterpret_cast<const float4*>(s_wa + (db * kPB + e) * ldw + col);
#pragma unroll
                        for (int e = 0; e < kPB; ++e)
                            acc[db * kPB + e] = fmaf(ha[c].x, w[e].x, fmaf(ha[c].y, w[e].y, fmaf(ha[c].z, w[e].z,
                                                fmaf(ha[c].w, w[e].w, acc[db * kPB + e]))));
                    }
                }
            }
            if (col < a.Hc) {
                const float4 w = *reinterpret_cast<const float4*>(s_wc + col);
                v_fused = fmaf(hc[c].x, w.x, fmaf(hc[c].y, w.y, fmaf(hc[c].z, w.z, fmaf(hc[c].w, w.w, v_fused))));
            }
        }
        LOSS_STAMP(2);
        // fold over the 32 lanes by recursive halving: at every step a lane keeps half of its values and trades the
        // other half with its partner, so 32 value slots cost 16+8+4+2+1 shuffles and lane l ends with the total of
        // slot l (slots 0..23: actor outputs, slot 24: the critic output)
        float v32[32];
#pragma unroll
        for (int d = 0; d < 32; ++d) v32[d] = d < kFusedMaxPred ? acc[d] : (d == kFusedMaxPred ? v_fused : 0.f);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const bool up = (lane & o) != 0;
#pragma unroll
            for (int k = 0; k < o; ++k) {
                const float send = up ? v32[k] : v32[k + o];
                const float keep = up ? v32[k + o] : v32[k];
                v32[k] = keep + __shfl_xor_sync(kFull, send, o);
            }
        }
        v_fused = __shfl_sync(kFull, v32[0], kFusedMaxPred) + s_b[a.pred_dim];
        if (gl < a.pred_dim) s_pred[smp * kFusedPredLd + gl] = v32[0] + s_b[gl];
        __syncwarp();                                                // the lanes of a sample share one warp
    }
    LOSS_STAMP(3);
    const float v = FUSED ? (live ? v_fused : 0.f) : (live ? a.critic_out[i] : 0.f);
    if (live && gl == 0) a.values[j] = v;                            // dataset.values[batch_idxs] = values (ppo.py:2340)
    float bad_value = isnan(v) ? 1.f : 0.f;

    const float* pred = FUSED ? s_pred + smp * kFusedPredLd : a.actor_out + int64_t(live ? i : 0) * a.pred_dim;
    float* dpred = a.d_actor_out + int64_t(live ? i : 0) * a.pred_dim;
    float* sdp = s_dpred + smp * kFusedPredLd;                       // FUSED: dL/d(actor out) kept for the head's dX
    actor_head_loss<FUSED>(a, gaussian, live, gl, j, pred, dpred, sdp, s_sd, adv, lp_old, inv_b, w_ent, clip_lo, clip_hi,
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

    // ---- fused heads, backward: dX of the two head layers times the activation derivative of the layer below ----
    if constexpr (FUSED) {
        __syncwarp();
        float dp[kFusedMaxPred];
#pragma unroll
        for (int d = 0; d < kFusedMaxPred; ++d) dp[d] = (d < a.pred_dim && live) ? sdp[d] : 0.f;
        const float gv = live ? dv1 * inv_b : 0.f;
        float* dza = a.dz_actor + int64_t(live ? i : 0) * a.Ha + 4 * gl;
        float* dzc = a.dz_critic + int64_t(live ? i : 0) * a.Hc + 4 * gl;
#pragma unroll
        for (int c = 0; c < kFusedMaxChunks; ++c) {
            const int col = 4 * (gl + kG * c);
            if (col < a.Ha) {
                float t[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int db = 0; db < kFusedMaxPred / kPB; ++db) {
                    if (db * kPB < a.pred_dim) {                     // padding rows of s_wa are zero
                        float4 w[kPB];
#pragma unroll
                        for (int e = 0; e < kPB; ++e) w[e] = *reinterpret_cast<const float4*>(s_wa + (db * kPB + e) * ldw + col);
#pragma unroll
                        for (int e = 0; e < kPB; ++e) {
                            t[0] = fmaf(dp[db * kPB + e], w[e].x, t[0]); t[1] = fmaf(dp[db * kPB + e], w[e].y, t[1]);
                            t[2] = fmaf(dp[db * kPB + e], w[e].z, t[2]); t[3] = fmaf(dp[db * kPB + e], w[e].w, t[3]);
                        }
                    }
                }
                const float y[4] = {ha[c].x, ha[c].y, ha[c].z, ha[c].w};
                act_bwd4(t, y, a.act);
                if (live) *reinterpret_cast<float4*>(dza + 4 * kG * c) = make_float4(t[0], t[1], t[2], t[3]);
            }
            if (col < a.Hc) {
                const float4 w = *reinterpret_cast<const float4*>(s_wc + col);
                float t[4] = {gv * w.x, gv * w.y, gv * w.z, gv * w.w};
                const float y[4] = {hc[c].x, hc[c].y, hc[c].z, hc[c].w};
                act_bwd4(t, y, a.act);
                if (live) *reinterpret_cast<float4*>(dzc + 4 * kG * c) = make_float4(t[0], t[1], t[2], t[3]);
            }
        }
    }

    LOSS_STAMP(5);
    // ---------------- CTA reduction (fp64, fixed order) ----------------
    // one warp per sample: lane 0 holds the sample's scalars, lane l holds d(loss)/d(std) of dims l, l + 32
    static_assert(kG == 32, "the reduction below assumes one warp per sample");
    const int n_extra = gaussian ? a.act_dim : 0;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) s_red[warp][k] = double(sc[k]);
    }
    if (gaussian) {
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) s_red[warp][kLossScalars + lane + k * kG] = double(dsd[k]);
    }
    __syncthreads();
    const int n_vals = kLossScalars + n_extra;
    double* part = reinterpret_cast<double*>(a.partials);
    if (tid < n_vals) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kLossThreads / 32; ++w) t += s_red[w][tid];
        part[size_t(blockIdx.x) * kPartialStride + tid] = t;
    }
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
    // thread (slot = tid % 32, subset = tid / 32) sums CTAs subset, subset + 8, ... for values slot, slot + 32, slot + 64
    // (all loads independent and in flight at once); the 8 subsets are then added in a fixed order
    {
        constexpr int kSub = kLossThreads / 32, kSlots = (kPartialStride + 31) / 32;
        double acc3[kSlots];
#pragma unroll
        for (int q = 0; q < kSlots; ++q) acc3[q] = 0.0;
        for (unsigned b = warp; b < gridDim.x; b += kSub) {
#pragma unroll
            for (int q = 0; q < kSlots; ++q) {
                const int vi = lane + 32 * q;
                if (vi < n_vals) acc3[q] += __ldcg(&part[size_t(b) * kPartialStride + vi]);
            }
        }
#pragma unroll
        for (int q = 0; q < kSlots; ++q) {
            const int vi = lane + 32 * q;
            if (vi < kPartialStride) s_red[warp][vi] = acc3[q];
        }
    }
    __syncthreads();
    __shared__ double s_sq[kLossThreads / 32];
    double my_sq = 0.0;
    if (tid < n_vals) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kLossThreads / 32; ++w) t += s_red[w][tid];
        s_tot[tid] = t;
        if (tid >= kLossScalars) {
            const float gls = float(t) * s_dsd[tid - kLossScalars];
            a.d_log_std[tid - kLossScalars] = gls;
            for (int q = 0; q < a.n_mirror; ++q)
                *reinterpret_cast<float*>(reinterpret_cast<char*>(a.d_log_std + (tid - kLossScalars)) + a.mirror_delta[q]) = gls;
            my_sq = double(gls) * double(gls);
        }
    }
    my_sq = warp_sum(my_sq);
    LOSS_STAMP(9);
    if (lane == 0) s_sq[warp] = my_sq;
    __syncthreads();
    if (tid == 0 && a.sq_log_std) {                        // sum of squares of d(log_std) for the gradient-norm clip
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < kLossThreads / 32; ++k) t += s_sq[k];
        *a.sq_log_std = t;
    }
    __syncthreads();
    if (tid == 0) {
        const double nb = double(a.batch);
        const float actor_mean = float(s_tot[LS_ACTOR] / nb);
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
        const double e0 = a.epoch_stats[PPOAF_ST_ACTOR_LOSS], e1 = a.epoch_stats[PPOAF_ST_CRITIC_LOSS];
        const double e2 = a.epoch_stats[PPOAF_ST_ENTROPY], e3 = a.epoch_stats[PPOAF_ST_KL];
        const double e4 = a.epoch_stats[PPOAF_ST_COUNTER], e5 = a.epoch_stats[PPOAF_ST_BAD_RATIO];
        const double e6 = a.epoch_stats[PPOAF_ST_BAD_VALUE];            // seven independent loads, then the stores
        a.epoch_stats[PPOAF_ST_ACTOR_LOSS] = e0 + double(actor_mean);
        a.epoch_stats[PPOAF_ST_CRITIC_LOSS] = e1 + double(critic_mean);
        if (w_ent != 0.f) a.epoch_stats[PPOAF_ST_ENTROPY] = e2 + double(float(s_tot[LS_ENTROPY] / nb));
        a.epoch_stats[PPOAF_ST_KL] = e3 + double(float(s_tot[LS_KL] / nb));
        a.epoch_stats[PPOAF_ST_COUNTER] = e4 + 1.0;
        a.epoch_stats[PPOAF_ST_BAD_RATIO] = e5 + s_tot[LS_BAD_RATIO];
        a.epoch_stats[PPOAF_ST_BAD_VALUE] = e6 + s_tot[LS_BAD_VALUE];
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

// ---- stand-alone head evaluation (PPOPolicy.evaluate's distribution half, policies/ppo_policy.py:939-950) ----
namespace ppoaf {

__global__ void head_evaluate_kernel(int head, const float* __restrict__ actor_out, int pred_dim,
                                     const float* __restrict__ log_std, float min_std, const void* __restrict__ actions,
                                     int act_dim, int n_rows, float* __restrict__ lp_out, float* __restrict__ ent_out) {
    __shared__ float s_sd[kMaxAct];
    const bool gaussian = head == PPOAF_HEAD_GAUSSIAN_TANH;
    if (gaussian && threadIdx.x < act_dim) s_sd[threadIdx.x] = fmaxf(softplus_torch(log_std[threadIdx.x]), min_std);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    float lp = 0.f, ent = 0.f;
    if (gaussian) {
        const float* x = reinterpret_cast<const float*>(actions) + int64_t(i) * act_dim;
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
        lp = nsum - slog;
        ent = -(ensum - eslog);
    } else {
        const int action = int(reinterpret_cast<const int64_t*>(actions)[int64_t(i) * act_dim]);
        float mx = pred[0];
        for (int c = 1; c < pred_dim; ++c) mx = fmaxf(mx, pred[c]);
        float se = 0.f;
        for (int c = 0; c < pred_dim; ++c) se += expf(pred[c] - mx);
        float S = 0.f;
        for (int c = 0; c < pred_dim; ++c) S += expf(pred[c] - mx) / se;
        const float ceps = 1.1920928955078125e-07f;
        float h = 0.f;
        for (int c = 0; c < pred_dim; ++c) {
            const float pn = (expf(pred[c] - mx) / se) / S;
            const float l = logf(fminf(fmaxf(pn, ceps), 1.f - ceps));
            h += pn * l;
            if (c == action) lp = l;
        }
        ent = -h;
    }
    lp_out[i] = lp;
    if (ent_out) ent_out[i] = ent;
}

}  // namespace ppoaf

namespace ppoaf {

// Rollout-time sampling (PPOPolicy.get_rollout_actions, policies/ppo_policy.py:729-794).  The random draws come from the
// HOST generator in the order the reference's CPU sampling consumes them (`noise`), so the actions are the reference's
// actions; everything else -- scaling by std, tanh squashing, range mapping, log-prob -- happens here.
//   Gaussian:    noise = N(0,1) [n, act_dim];  raw = noise * std + mean  (torch.normal: mul_ then add_)
//                action = tanh(raw), mapped to [min, max] when given (distributions.py:560-610); log-prob :518-558
//   Categorical: noise = Exp(1) [n, pred];  sample = argmax(p / noise)  (aten multinomial, one draw); log-prob :223-249
__global__ void head_sample_kernel(int head, const float* __restrict__ actor_out, int pred_dim,
                                   const float* __restrict__ log_std, float min_std, const float* __restrict__ noise,
                                   const float* __restrict__ dist_min, const float* __restrict__ dist_max, int act_dim,
                                   int n_rows, void* __restrict__ raw_out, void* __restrict__ act_out,
                                   float* __restrict__ lp_out) {
    __shared__ float s_sd[kMaxAct];
    const bool gaussian = head == PPOAF_HEAD_GAUSSIAN_TANH;
    if (gaussian && threadIdx.x < act_dim) s_sd[threadIdx.x] = fmaxf(softplus_torch(log_std[threadIdx.x]), min_std);
    __syncthreads();
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    if (gaussian) {
        const float* z = noise + int64_t(i) * act_dim;
        float* raw = reinterpret_cast<float*>(raw_out) + int64_t(i) * act_dim;
        float* act = reinterpret_cast<float*>(act_out) + int64_t(i) * act_dim;
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
    } else {
        const float* q = noise + int64_t(i) * pred_dim;
        float S = 0.f;
        for (int c = 0; c < pred_dim; ++c) S += pred[c];
        int best = 0;
        float best_v = -INFINITY, best_p = 0.f;
        for (int c = 0; c < pred_dim; ++c) {
            const float pn = pred[c] / S;
            const float v = pn / q[c];
            if (v > best_v) { best_v = v; best = c; best_p = pn; }          // first maximum, like argmax
        }
        reinterpret_cast<int64_t*>(raw_out)[i] = best;
        reinterpret_cast<int64_t*>(act_out)[i] = best;
        lp_out[i] = logf(fminf(fmaxf(best_p, kCatEps), 1.f - kCatEps));
    }
}

}  // namespace ppoaf

extern "C" int ppoaf_head_sample(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                                 float min_std, const float* noise, const float* dist_min, const float* dist_max,
                                 int32_t act_dim, int32_t n_rows, void* raw_action_out, void* action_out,
                                 float* log_prob_out, void* stream) {
    using namespace ppoaf;
    PPOAF_CHECK_ARG(head == PPOAF_HEAD_GAUSSIAN_TANH || head == PPOAF_HEAD_CATEGORICAL, "ppoaf_head_sample: unknown head");
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= kMaxAct && pred_dim >= 1 && pred_dim <= kMaxAct,
                    "ppoaf_head_sample: widths must be in [1, %d]", kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0 && noise != nullptr, "ppoaf_head_sample: bad arguments");
    PPOAF_CHECK_ARG((dist_min == nullptr) == (dist_max == nullptr), "ppoaf_head_sample: give both range bounds or neither");
    if (n_rows == 0) return 0;
    head_sample_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        head, actor_out, pred_dim, log_std, min_std, noise, dist_min, dist_max, act_dim, n_rows, raw_action_out, action_out,
        log_prob_out);
    PPOAF_CHECK_LAUNCH("ppoaf_head_sample");
    return 0;
}

extern "C" int ppoaf_head_evaluate(int32_t head, const float* actor_out, int32_t pred_dim, const float* log_std,
                                   float min_std, const void* actions, int32_t act_dim, int32_t n_rows,
                                   float* log_prob_out, float* entropy_out, void* stream) {
    using namespace ppoaf;
    PPOAF_CHECK_ARG(head == PPOAF_HEAD_GAUSSIAN_TANH || head == PPOAF_HEAD_CATEGORICAL, "ppoaf_head_evaluate: unknown head");
    PPOAF_CHECK_ARG(act_dim >= 1 && act_dim <= kMaxAct && pred_dim >= 1 && pred_dim <= kMaxAct,
                    "ppoaf_head_evaluate: widths must be in [1, %d]", kMaxAct);
    PPOAF_CHECK_ARG(n_rows >= 0, "ppoaf_head_evaluate: n_rows < 0");
    if (n_rows == 0) return 0;
    head_evaluate_kernel<<<(n_rows + 127) / 128, 128, 0, (cudaStream_t)stream>>>(
        head, actor_out, pred_dim, log_std, min_std, actions, act_dim, n_rows, log_prob_out, entropy_out);
    PPOAF_CHECK_LAUNCH("ppoaf_head_evaluate");
    return 0;
}

// ---- the multi-categorical head on its own (PPOAF_HEAD_MULTI_CATEGORICAL): one thread per row, sections in order ----
namespace ppoaf {

__global__ void multi_categorical_evaluate_kernel(const float* __restrict__ actor_out, int pred_dim,
                                                  unsigned long long ends, const int64_t* __restrict__ actions,
                                                  int n_sections, int n_rows, float* __restrict__ lp_out,
                                                  float* __restrict__ ent_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* pred = actor_out + int64_t(i) * pred_dim;
    const int64_t* act = actions + int64_t(i) * n_sections;
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

// probs: the softmax of the whole row; noise: section k's Exp(1) block [n_rows, n_k] starts at n_rows * o_k
__global__ void multi_categorical_sample_kernel(const float* __restrict__ probs, int pred_dim, unsigned long long ends,
                                                const float* __restrict__ noise, int n_sections, int n_rows,
                                                int64_t* __restrict__ act_out, float* __restrict__ lp_out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_rows) return;
    const float* p = probs + int64_t(i) * pred_dim;
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
        act_out[int64_t(i) * n_sections + k] = best;
        lp += logf(fminf(fmaxf(best_p, kCatEps), 1.f - kCatEps));
        o = c + 1;
        ++k;
    }
    lp_out[i] = lp;
}

}  // namespace ppoaf

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
        probs, pred_dim, ends, noise, n_sections, n_rows, actions_out_i64, log_prob_out);
    PPOAF_CHECK_LAUNCH("ppoaf_multi_categorical_sample");
    return 0;
}
