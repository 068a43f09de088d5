// Pieces of the fused PPO loss shared by the stand-alone loss kernel (loss.cu) and the persistent whole-step kernel
// (fused_step.cu): widths, the partial-sum layout and the action-head arithmetic (reference ppo.py:2342-2410 with
// networks/distributions.py:491-558, 694 and torch's Normal / Categorical).
#pragma once
#include "internal.h"

namespace ppoaf {

constexpr int kMaxAct = 64;
constexpr int kG = 32;                      // lanes that share one sample: one warp (each lane owns dims l, l+32)
constexpr int kPerLane = kMaxAct / kG;      // 2
constexpr int kLossThreads = 256;           // 8 samples per CTA
constexpr int kSamplesPerBlock = kLossThreads / kG;
enum { LS_ACTOR = 0, LS_CRITIC, LS_CRITIC_CLIPPED, LS_ENTROPY, LS_KL, LS_BAD_RATIO, LS_BAD_VALUE, kLossScalars };
constexpr int kPartialStride = kLossScalars + kMaxAct;

// fused head layers: widths the register-resident path supports
constexpr int kFusedMaxPred = 24;           // actor head outputs
constexpr int kFusedMaxChunks = 2;          // hidden width <= 256: lane gl owns columns 4 (gl + 32 c) .. + 3
constexpr int kFusedPredLd = kFusedMaxPred + 1;
constexpr int kPB = 8;                      // head rows are processed in blocks of 8 independent rows
constexpr int kFusedStageSlots = kFusedMaxPred * (kG * kFusedMaxChunks) / 256;   // float4 per thread to stage W_actor


constexpr float kLogSqrt2Pi = 0.91893853320467274178f;
constexpr float kCatEps = 1.1920928955078125e-07f;   // torch.finfo(float32).eps

__device__ __forceinline__ float softplus_torch(float x) { return x > 20.f ? x : log1pf(expf(x)); }

__device__ __forceinline__ float critic_term(float v, float target, int use_huber, float& dv) {
    const float d = v - target;
    if (use_huber) {
        const float delta = 10.f, ad = fabsf(d);
        if (ad < delta) { dv = d; return 0.5f * d * d; }
        dv = d > 0.f ? delta : -delta;
        return delta * (ad - 0.5f * delta);
    }
    dv = 2.f * d;
    return d * d;
}

// sum / max over the kG lanes that share a sample (lanes are contiguous inside a warp)
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
    for (int o = kG / 2; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
    for (int o = kG / 2; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(kFull, v, o));
    return v;
}

// Multi-categorical section table (bit c set: column c ends a section).  For a column c < 64: first column of its
// section, last column of its section (-1 past the last section) and the section's index.
__device__ __forceinline__ int section_start(unsigned long long ends, int c) {
    const unsigned long long below = ends & ((1ull << c) - 1ull);
    return below ? 64 - __clzll((long long)below) : 0;
}
__device__ __forceinline__ int section_end(unsigned long long ends, int c) { return __ffsll((long long)(ends >> c << c)) - 1; }
__device__ __forceinline__ int section_index(unsigned long long ends, int c) { return __popcll(ends & ((1ull << c) - 1ull)); }

// Per-section sums over the kG lanes of one sample: out[k] = sum of v over the section that column gl + k kG belongs
// to (st / en: first / last column of that section).  A segmented inclusive scan of each half of the row (a lane adds
// its neighbour's partial sum only while that neighbour lies in the same section), the second half continuing the
// section column 31 leaves open, then every lane reads the scan at its section's last column.  A table of one section
// takes the Categorical head's whole-row sum instead (same order), so MultiDiscrete([n]) reproduces Discrete(n) exactly.
__device__ __forceinline__ void section_sum(const float (&v)[kPerLane], const int (&st)[kPerLane],
                                            const int (&en)[kPerLane], int gl, bool one_section,
                                            float (&out)[kPerLane]) {
    if (one_section) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) t += v[k];
        t = group_sum(t);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) out[k] = t;
        return;
    }
    float x[kPerLane];
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) x[k] = v[k];
#pragma unroll
    for (int o = 1; o < kG; o <<= 1) {
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const float y = __shfl_up_sync(kFull, x[k], o);
            if (gl >= o && gl - o + k * kG >= st[k]) x[k] += y;
        }
    }
    static_assert(kPerLane == 2, "the carry below joins two halves of the row");
    const float carry = __shfl_sync(kFull, x[0], kG - 1);
    if (st[1] < kG) x[1] += carry;
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) {
        const int e = en[k] < 0 ? 0 : en[k];
        const float lo = __shfl_sync(kFull, x[0], e & (kG - 1)), hi = __shfl_sync(kFull, x[1], e & (kG - 1));
        out[k] = e >= kG ? hi : lo;
    }
}

// Action-head part of the loss for one sample shared by the 32 lanes of a warp (lane gl owns dims gl, gl + 32):
// log-prob, entropy, ratio, clipped surrogate and their gradients w.r.t. the head outputs (written to dpred, and
// to sdp when the head layer itself is fused) and w.r.t. std (dsd).  Lane 0 receives the sample's scalars in sc.
template <bool FUSED>
__device__ __forceinline__ void actor_head_loss(const LossArgs& a, bool gaussian, bool live, int gl, int64_t j,
                                                const float* pred, float* dpred, float* sdp, const float* s_sd,
                                                float adv, float lp_old, float inv_b, float w_ent, float clip_lo,
                                                float clip_hi, float (&sc)[kLossScalars], float (&dsd)[kPerLane],
                                                float& bad_value) {
    float lp = 0.f, ent = 0.f;
    if (gaussian) {
        const float* x = reinterpret_cast<const float*>(a.raw_actions) + j * a.act_dim;
        float mu[kPerLane], z[kPerLane], on[kPerLane], one[kPerLane], thm[kPerLane];
        float nsum = 0.f, slog = 0.f, ensum = 0.f, eslog = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int d = gl + k * kG;
            mu[k] = z[k] = on[k] = one[k] = thm[k] = 0.f;
            if (d < a.act_dim && live) {
                const float sd = s_sd[d], xd = x[d];
                mu[k] = pred[d];
                z[k] = xd - mu[k];
                bad_value = fmaxf(bad_value, isnan(mu[k]) ? 1.f : 0.f);
                const float lsd = logf(sd);
                const float nl = -(z[k] * z[k]) / (2.f * (sd * sd)) - lsd - kLogSqrt2Pi;   // Normal.log_prob
                nsum += fminf(fmaxf(nl, -100.f), 100.f);
                on[k] = (nl >= -100.f && nl <= 100.f) ? 1.f : 0.f;
                const float th = tanhf(xd);
                slog += logf(fmaxf(1.f - th * th, 1e-6f));
                const float nle = -lsd - kLogSqrt2Pi;                                     // log N(mu; mu, sd)
                ensum += fminf(fmaxf(nle, -100.f), 100.f);
                one[k] = (nle >= -100.f && nle <= 100.f) ? 1.f : 0.f;
                thm[k] = tanhf(mu[k]);
                eslog += logf(fmaxf(1.f - thm[k] * thm[k], 1e-6f));
            }
        }
        lp = group_sum(nsum) - group_sum(slog);
        ent = -(group_sum(ensum) - group_sum(eslog));                 // entropy = -log_prob(mean) (:694)
        const float ratio = expf(lp - lp_old);
        const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, clip_lo), clip_hi) * adv;
        // d(-min(s1,s2))/d lp flows through s1 when s1 <= s2 (on a tie both branches carry half and the
        // clamp passes its half exactly when rho is inside the clip range, which the tie implies)
        const float g_lp = (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
        const float g_ent = -w_ent * inv_b;                           // dL/dH_i
        if (gl == 0 && live) {
            sc[LS_ACTOR] = -fminf(s1, s2);
            sc[LS_KL] = lp_old - lp;
            sc[LS_ENTROPY] = ent;
            sc[LS_BAD_RATIO] = (isnan(ratio) || isinf(ratio)) ? 1.f : 0.f;
        }
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int d = gl + k * kG;
            if (d < a.act_dim && live) {
                const float sd = s_sd[d], var = sd * sd;
                const float tmask = (1.f - thm[k] * thm[k] >= 1e-6f) ? 1.f : 0.f;
                // dlp/dmu = z/var ; dH/dmu = -2 tanh(mu)
                const float gd = g_lp * on[k] * (z[k] / var) + g_ent * tmask * (-2.f * thm[k]);
                dpred[d] = gd;
                if constexpr (FUSED) sdp[d] = gd;
                // dlp/dsd = z^2/sd^3 - 1/sd ; dH/dsd = 1/sd
                dsd[k] = g_lp * on[k] * ((z[k] * z[k]) / (var * sd) - 1.f / sd) + g_ent * one[k] * (1.f / sd);
            }
        }
    } else if (a.head == PPOAF_HEAD_MULTI_CATEGORICAL) {
        // softmax over the whole row (as for Categorical), then one Categorical(probs) per section: the Categorical
        // arithmetic with the renormaliser S and the sum of G p taken per section (section_sum)
        const unsigned long long ends = a.section_ends;
        const bool one_section = (ends & (ends - 1ull)) == 0ull;
        const int n = a.pred_dim;
        const int64_t* acts = reinterpret_cast<const int64_t*>(a.raw_actions) + j * a.act_dim;
        float p[kPerLane], pn[kPerLane], lg[kPerLane];
        int st[kPerLane], en[kPerLane];
        bool hit[kPerLane];
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            st[k] = section_start(ends, c);
            en[k] = section_end(ends, c);
            p[k] = (c < n) ? pred[c] : -INFINITY;
            hit[k] = live && c < n && c - st[k] == int(acts[section_index(ends, c)]);
            if (c < n) bad_value = fmaxf(bad_value, isnan(p[k]) ? 1.f : 0.f);
            mx = fmaxf(mx, p[k]);
        }
        mx = group_max(mx);
        float se = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            p[k] = (c < n) ? expf(p[k] - mx) : 0.f;
            se += p[k];
        }
        se = group_sum(se);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) p[k] = p[k] / se;
        float S[kPerLane];
        section_sum(p, st, en, gl, one_section, S);
        float h = 0.f, lpa = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            pn[k] = lg[k] = 0.f;
            if (c < n) {
                pn[k] = p[k] / S[k];
                lg[k] = logf(fminf(fmaxf(pn[k], kCatEps), 1.f - kCatEps));
                h += pn[k] * lg[k];
                if (hit[k]) lpa += lg[k];
            }
        }
        lp = group_sum(lpa);                                                    // sums over the sections
        ent = -group_sum(h);
        const float ratio = expf(lp - lp_old);
        const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, clip_lo), clip_hi) * adv;
        const float g_lp = (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
        const float g_ent = -w_ent * inv_b;
        if (gl == 0 && live) {
            sc[LS_ACTOR] = -fminf(s1, s2);
            sc[LS_KL] = lp_old - lp;
            sc[LS_ENTROPY] = ent;
            sc[LS_BAD_RATIO] = (isnan(ratio) || isinf(ratio)) ? 1.f : 0.f;
        }
        // G_c = dL/d pn_c ; pn = p / S_k ; p = softmax(z)
        float G[kPerLane], gp[kPerLane];
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            G[k] = gp[k] = 0.f;
            if (c < n) {
                const float q = fminf(fmaxf(pn[k], kCatEps), 1.f - kCatEps);
                const float mask = (pn[k] >= kCatEps && pn[k] <= 1.f - kCatEps) ? 1.f : 0.f;
                const float dlg = (hit[k] ? g_lp : 0.f) + g_ent * (-pn[k]);
                G[k] = g_ent * (-lg[k]) + dlg * mask / q;
                gp[k] = G[k] * p[k];
            }
        }
        float gdotp[kPerLane];
        section_sum(gp, st, en, gl, one_section, gdotp);
        float dpdotp = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            if (c < n) {
                G[k] = G[k] / S[k] - gdotp[k] / (S[k] * S[k]);                  // dL/dp_c
                dpdotp += G[k] * p[k];
            }
        }
        dpdotp = group_sum(dpdotp);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            if (c < n && live) {
                const float gd = p[k] * (G[k] - dpdotp);
                dpred[c] = gd;
                if constexpr (FUSED) sdp[c] = gd;
            }
        }
    } else {
        const int n = a.pred_dim;
        const int action = live ? int(reinterpret_cast<const int64_t*>(a.raw_actions)[j * a.act_dim]) : 0;
        float p[kPerLane], pn[kPerLane], lg[kPerLane];
        float mx = -INFINITY;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            p[k] = (c < n) ? pred[c] : -INFINITY;
            if (c < n) bad_value = fmaxf(bad_value, isnan(p[k]) ? 1.f : 0.f);
            mx = fmaxf(mx, p[k]);
        }
        mx = group_max(mx);
        float se = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            p[k] = (c < n) ? expf(p[k] - mx) : 0.f;
            se += p[k];
        }
        se = group_sum(se);
        float S = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) { p[k] = p[k] / se; S += p[k]; }       // softmax inside the actor (:1045)
        S = group_sum(S);
        float h = 0.f, lpa = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            pn[k] = p[k] / S;                                                       // Categorical renormalises probs
            lg[k] = logf(fminf(fmaxf(pn[k], kCatEps), 1.f - kCatEps));
            if (c < n) { h += pn[k] * lg[k]; if (c == action) lpa = lg[k]; }
        }
        lp = group_sum(lpa);
        ent = -group_sum(h);
        const float ratio = expf(lp - lp_old);
        const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, clip_lo), clip_hi) * adv;
        const float g_lp = (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
        const float g_ent = -w_ent * inv_b;
        if (gl == 0 && live) {
            sc[LS_ACTOR] = -fminf(s1, s2);
            sc[LS_KL] = lp_old - lp;
            sc[LS_ENTROPY] = ent;
            sc[LS_BAD_RATIO] = (isnan(ratio) || isinf(ratio)) ? 1.f : 0.f;
        }
        // G_c = dL/d pn_c ; pn = p / S ; p = softmax(z)
        float G[kPerLane];
        float gdotp = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            G[k] = 0.f;
            if (c < n) {
                const float q = fminf(fmaxf(pn[k], kCatEps), 1.f - kCatEps);
                const float mask = (pn[k] >= kCatEps && pn[k] <= 1.f - kCatEps) ? 1.f : 0.f;
                const float dlg = (c == action ? g_lp : 0.f) + g_ent * (-pn[k]);
                G[k] = g_ent * (-lg[k]) + dlg * mask / q;
                gdotp += G[k] * p[k];
            }
        }
        gdotp = group_sum(gdotp);
        float dpdotp = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            G[k] = G[k] / S - gdotp / (S * S);                                      // dL/dp_c
            dpdotp += G[k] * p[k];
        }
        dpdotp = group_sum(dpdotp);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            if (c < n && live) {
                const float gd = p[k] * (G[k] - dpdotp);
                dpred[c] = gd;
                if constexpr (FUSED) sdp[c] = gd;
            }
        }
    }
}

}  // namespace ppoaf
