// The per-sample PPO loss, shared by the stand-alone loss kernel (loss.cu) and the LOSS phase of the persistent
// whole-step kernel (fused_step.cu): widths, the partial-sum layout, the action-head arithmetic (reference
// ppo.py:2342-2410 with networks/distributions.py:491-558, 694 and torch's Normal / Categorical / Bernoulli), the fused head layers
// and the reductions.  The two kernels differ only in how they load their inputs and how their CTAs meet.
#pragma once
#include "internal.h"

namespace ppoaf {

constexpr int kMaxAct = kMaxNarrowHead;      // wider Categorical / Gaussian rows: the wide kernels of loss.cu
constexpr int kG = 32;                     // lanes that share one sample: one warp (each lane owns dims l, l+32)
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
// (the Categorical head, MultiDiscrete([n])) takes a plain whole-row sum instead.
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

// Bernoulli (MultiBinary) columns, torch's Bernoulli(probs = sigmoid(z)) restated (DESIGN §4): q = clamp(p, eps,
// 1 - eps), l = log q - log1p(-q); log_prob(x) = logsigmoid(l) - (1 - x) l, entropy = (1 - p) l - logsigmoid(l)
__device__ __forceinline__ float sigmoid_f(float z) { return 1.f / (1.f + expf(-z)); }
__device__ __forceinline__ float bernoulli_logit(float p) {
    const float q = fminf(fmaxf(p, kCatEps), 1.f - kCatEps);
    return logf(q) - log1pf(-q);
}
__device__ __forceinline__ float log_sigmoid(float l) { return fminf(l, 0.f) - log1pf(expf(-fabsf(l))); }

// std = max(softplus(log_std), min_std) (distributions.py:514-515) and dstd = d std / d log_std (torch's max splits the
// gradient evenly on a tie)
__device__ __forceinline__ float std_of_log_std(float ls, float min_std, float& dstd) {
    const float sp = softplus_torch(ls);
    const float sig = ls > 20.f ? 1.f : 1.f / (1.f + expf(-ls));
    dstd = sp > min_std ? sig : (sp == min_std ? 0.5f * sig : 0.f);
    return fmaxf(sp, min_std);
}

// Clipped surrogate of one sample from its log-prob and entropy: returns dL/d lp; `first` (lane 0 of a live sample)
// records the sample's scalars.  d(-min(s1,s2))/d lp flows through s1 when s1 <= s2 (on a tie both branches carry half
// and the clamp passes its half exactly when rho is inside the clip range, which the tie implies).
__device__ __forceinline__ float ppo_surrogate(float lp, float ent, float lp_old, float adv, float inv_b, float clip_lo,
                                               float clip_hi, bool first, float (&sc)[kLossScalars]) {
    const float ratio = expf(lp - lp_old);
    const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, clip_lo), clip_hi) * adv;
    if (first) {
        sc[LS_ACTOR] = -fminf(s1, s2);
        sc[LS_KL] = lp_old - lp;
        sc[LS_ENTROPY] = ent;
        sc[LS_BAD_RATIO] = (isnan(ratio) || isinf(ratio)) ? 1.f : 0.f;
    }
    return (s1 <= s2) ? -adv * ratio * inv_b : 0.f;
}

// Action-head part of the loss for one sample shared by the 32 lanes of a warp (lane gl owns dims gl, gl + 32):
// log-prob, entropy, ratio, clipped surrogate and their gradients w.r.t. the head outputs (written to dpred, and
// to sdp when the head layer itself is fused) and w.r.t. std (dsd, Gaussian head only).  Lane 0 receives the sample's
// scalars in sc.  head: PPOAF_HEAD_*.
template <bool FUSED>
__device__ __forceinline__ void actor_head_loss(const LossArgs& a, int head, bool live, int gl, int64_t j,
                                                const float* pred, float* dpred, float* sdp, const float* s_sd,
                                                float adv, float lp_old, float inv_b, float w_ent, float clip_lo,
                                                float clip_hi, float (&sc)[kLossScalars], float (&dsd)[kPerLane],
                                                float& bad_value) {
    const float g_ent = -w_ent * inv_b;                               // dL/dH_i
    if (head == PPOAF_HEAD_GAUSSIAN_TANH) {
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
        const float lp = group_sum(nsum) - group_sum(slog);
        const float ent = -(group_sum(ensum) - group_sum(eslog));    // entropy = -log_prob(mean) (:694)
        const float g_lp = ppo_surrogate(lp, ent, lp_old, adv, inv_b, clip_lo, clip_hi, gl == 0 && live, sc);
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
    } else if (head == PPOAF_HEAD_BERNOULLI) {
        // independent columns p = sigmoid(z) (bernoulli_logit / log_sigmoid above); log-prob and entropy are the sums
        // over the act_dim columns.  Backward with s = sigmoid(l) and m = [eps <= p <= 1 - eps] (the clamp passes the
        // gradient on its bounds): dL/dp = g_lp (x - s) m / (q (1 - q)) + g_ent ((s - p) m / (q (1 - q)) - l), then
        // dL/dz = dL/dp p (1 - p).
        const float* x = reinterpret_cast<const float*>(a.raw_actions) + j * a.act_dim;
        float p[kPerLane], l[kPerLane], xv[kPerLane];
        float lpa = 0.f, h = 0.f;
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            p[k] = l[k] = xv[k] = 0.f;
            if (c < a.act_dim && live) {
                const float zc = pred[c];
                bad_value = fmaxf(bad_value, isnan(zc) ? 1.f : 0.f);
                xv[k] = x[c];
                p[k] = sigmoid_f(zc);
                l[k] = bernoulli_logit(p[k]);
                const float ls = log_sigmoid(l[k]);
                lpa += ls - (1.f - xv[k]) * l[k];
                h += (1.f - p[k]) * l[k] - ls;
            }
        }
        const float lp = group_sum(lpa);
        const float ent = group_sum(h);
        const float g_lp = ppo_surrogate(lp, ent, lp_old, adv, inv_b, clip_lo, clip_hi, gl == 0 && live, sc);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) {
            const int c = gl + k * kG;
            if (c < a.act_dim && live) {
                const float q = fminf(fmaxf(p[k], kCatEps), 1.f - kCatEps);
                const float r = (p[k] >= kCatEps && p[k] <= 1.f - kCatEps) ? 1.f / (q * (1.f - q)) : 0.f;
                const float s = sigmoid_f(l[k]);
                const float gp = g_lp * (xv[k] - s) * r + g_ent * ((s - p[k]) * r - l[k]);
                const float gd = gp * (p[k] * (1.f - p[k]));
                dpred[c] = gd;
                if constexpr (FUSED) sdp[c] = gd;
            }
        }
    } else {
        // (multi-)categorical: softmax over the whole row (:1045), then one Categorical(probs) per section, which
        // renormalises its probs: the renormaliser S and the sum of G p are taken per section (section_sum).  The
        // Categorical head is the table of one section.
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
        const float lp = group_sum(lpa);                                        // sums over the sections
        const float ent = -group_sum(h);
        const float g_lp = ppo_surrogate(lp, ent, lp_old, adv, inv_b, clip_lo, clip_hi, gl == 0 && live, sc);
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
    }
}

// Shared-memory layout of the fused head layers (loss_head_fusable): W_actor [prows][ldw] (rows padded with zeros to
// whole blocks of kPB; the pitch Ha + 4 puts the rows on distinct bank groups) | W_critic [Hc] | b_actor, b_critic
// [pred + 1, padded to 4] | actor outputs and their gradients, [kSamplesPerBlock][kFusedPredLd] each
struct HeadSmem {
    int prows, ldw;
    float *wa, *wc, *b, *pred, *dpred;
    __device__ __forceinline__ HeadSmem(const LossArgs& a, float* s)
        : prows((a.pred_dim + kPB - 1) / kPB * kPB), ldw(a.Ha + 4), wa(s), wc(wa + prows * ldw), b(wc + a.Hc),
          pred(b + ((a.pred_dim + 1 + 3) & ~3)), dpred(pred + kSamplesPerBlock * kFusedPredLd) {}
};

// Head layers, forward, for the sample of one warp (lane gl holds hidden columns 4 (gl + kG c) .. + 3 in ha / hc): every
// lane dots its columns with all head rows, then the 32 lanes fold their partial sums by recursive halving: at every
// step a lane keeps half of its values and trades the other half with its partner, so 32 value slots cost 16+8+4+2+1
// shuffles and lane l ends with the total of slot l (slots 0..23: actor outputs, slot 24: the critic output).  The
// actor outputs go to pred; returns the critic output.
__device__ __forceinline__ float head_forward(const LossArgs& a, const HeadSmem& s, const float4 (&ha)[kFusedMaxChunks],
                                              const float4 (&hc)[kFusedMaxChunks], int gl, float* pred) {
    float acc[kFusedMaxPred];
#pragma unroll
    for (int d = 0; d < kFusedMaxPred; ++d) acc[d] = 0.f;
    float v = 0.f;
#pragma unroll
    for (int c = 0; c < kFusedMaxChunks; ++c) {
        const int col = 4 * (gl + kG * c);
        if (col < a.Ha) {
#pragma unroll
            for (int db = 0; db < kFusedMaxPred / kPB; ++db) {
                if (db * kPB < a.pred_dim) {                         // uniform: whole blocks of independent rows
                    float4 w[kPB];
#pragma unroll
                    for (int e = 0; e < kPB; ++e) w[e] = *reinterpret_cast<const float4*>(s.wa + (db * kPB + e) * s.ldw + col);
#pragma unroll
                    for (int e = 0; e < kPB; ++e)
                        acc[db * kPB + e] = fmaf(ha[c].x, w[e].x, fmaf(ha[c].y, w[e].y, fmaf(ha[c].z, w[e].z,
                                            fmaf(ha[c].w, w[e].w, acc[db * kPB + e]))));
                }
            }
        }
        if (col < a.Hc) {
            const float4 w = *reinterpret_cast<const float4*>(s.wc + col);
            v = fmaf(hc[c].x, w.x, fmaf(hc[c].y, w.y, fmaf(hc[c].z, w.z, fmaf(hc[c].w, w.w, v))));
        }
    }
    static_assert(kG == 32 && kFusedMaxPred < 32, "the fold below gives one lane of the warp to every head output");
    float v32[32];
#pragma unroll
    for (int d = 0; d < 32; ++d) v32[d] = d < kFusedMaxPred ? acc[d] : (d == kFusedMaxPred ? v : 0.f);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const bool up = (gl & o) != 0;
#pragma unroll
        for (int k = 0; k < o; ++k) {
            const float send = up ? v32[k] : v32[k + o];
            const float keep = up ? v32[k + o] : v32[k];
            v32[k] = keep + __shfl_xor_sync(kFull, send, o);
        }
    }
    v = __shfl_sync(kFull, v32[0], kFusedMaxPred) + s.b[a.pred_dim];
    if (gl < a.pred_dim) pred[gl] = v32[0] + s.b[gl];
    __syncwarp();                                                    // the lanes of a sample share one warp
    return v;
}

// Head layers, backward: dX of the two head layers (dL/d actor outputs in dpred, dL/d value dv * inv_b) times the
// activation derivative of the layer below, stored to row `row` of dz_actor / dz_critic
__device__ __forceinline__ void head_backward(const LossArgs& a, const HeadSmem& s, const float4 (&ha)[kFusedMaxChunks],
                                              const float4 (&hc)[kFusedMaxChunks], const float* dpred, float dv,
                                              float inv_b, bool live, int gl, int64_t row) {
    __syncwarp();
    float dp[kFusedMaxPred];
#pragma unroll
    for (int d = 0; d < kFusedMaxPred; ++d) dp[d] = (d < a.pred_dim && live) ? dpred[d] : 0.f;
    const float gv = live ? dv * inv_b : 0.f;
    float* dza = a.dz_actor + row * a.Ha + 4 * gl;
    float* dzc = a.dz_critic + row * a.Hc + 4 * gl;
#pragma unroll
    for (int c = 0; c < kFusedMaxChunks; ++c) {
        const int col = 4 * (gl + kG * c);
        if (col < a.Ha) {
            float t[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
            for (int db = 0; db < kFusedMaxPred / kPB; ++db) {
                if (db * kPB < a.pred_dim) {                         // padding rows of s.wa are zero
                    float4 w[kPB];
#pragma unroll
                    for (int e = 0; e < kPB; ++e) w[e] = *reinterpret_cast<const float4*>(s.wa + (db * kPB + e) * s.ldw + col);
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
            const float4 w = *reinterpret_cast<const float4*>(s.wc + col);
            float t[4] = {gv * w.x, gv * w.y, gv * w.z, gv * w.w};
            const float y[4] = {hc[c].x, hc[c].y, hc[c].z, hc[c].w};
            act_bwd4(t, y, a.act);
            if (live) *reinterpret_cast<float4*>(dzc + 4 * kG * c) = make_float4(t[0], t[1], t[2], t[3]);
        }
    }
}

// ---- reductions of the loss (fp64, fixed order).  `bar` is the barrier of the kLossThreads threads that run them. ----
// CTA partials: lane 0 of warp w holds the scalars of the warp's samples, lane l their d loss / d std of dims l, l + 32;
// the CTA's sums of the first n_vals values go to slot blockIdx.x of part
template <class T, class Bar>
__device__ __forceinline__ void loss_cta_partials(const T (&sc)[kLossScalars], const T (&dsd)[kPerLane],
                                                  int n_vals, double (*s_red)[kPartialStride], double* part, Bar bar) {
    static_assert(kG == 32, "one warp per sample");
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) s_red[warp][k] = double(sc[k]);
    }
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) s_red[warp][kLossScalars + lane + k * kG] = double(dsd[k]);
    bar();
    if (tid < n_vals) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kLossThreads / 32; ++w) t += s_red[w][tid];
        part[size_t(blockIdx.x) * kPartialStride + tid] = t;
    }
}

// d(log_std) of dim d (the batch total of dL/d std times d std / d log_std), stored with its peer mirrors
__device__ __forceinline__ void store_d_log_std(const LossArgs& a, int d, float gls) {
    a.d_log_std[d] = gls;
    for (int q = 0; q < a.n_mirror; ++q)
        *reinterpret_cast<float*>(reinterpret_cast<char*>(a.d_log_std + d) + a.mirror_delta[q]) = gls;
}

// One CTA, after every CTA's partials are visible: totals -> s_tot, d(log_std) (and its peer mirrors) and the sum of
// squares of d(log_std) for the gradient-norm clip.  Thread (slot = tid % 32, subset = tid / 32) sums CTAs subset,
// subset + 8, ... for values slot, slot + 32, slot + 64 (all loads independent and in flight at once, from L2); the 8
// subsets are then added in a fixed order.  s_tot is complete on return.
template <class Bar>
__device__ __forceinline__ void loss_fold(const LossArgs& a, int n_vals, const float* s_dsd, double (*s_red)[kPartialStride],
                                          double* s_tot, double* s_sq, Bar bar) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const double* part = reinterpret_cast<const double*>(a.partials);
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
    bar();
    double my_sq = 0.0;
    if (tid < n_vals) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kLossThreads / 32; ++w) t += s_red[w][tid];
        s_tot[tid] = t;
        if (tid >= kLossScalars) {
            const float gls = float(t) * s_dsd[tid - kLossScalars];
            store_d_log_std(a, tid - kLossScalars, gls);
            my_sq = double(gls) * double(gls);
        }
    }
    my_sq = warp_sum(my_sq);
    if (lane == 0) s_sq[warp] = my_sq;
    bar();
    if (tid == 0 && a.sq_log_std) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < kLossThreads / 32; ++k) t += s_sq[k];
        *a.sq_log_std = t;
    }
}

// Epoch statistics of the minibatch from the totals (one thread); critic_mean: the mean critic loss the update used.
// w_ent is read by the caller, early: a load of a.hparams here would wait for the stores to a.epoch_stats it may alias.
__device__ __forceinline__ void add_epoch_stats(const LossArgs& a, const double* s_tot, float critic_mean, float w_ent) {
    const double nb = double(a.batch);
    const float actor_mean = float(s_tot[LS_ACTOR] / nb);
    double* es = a.epoch_stats;
    const double e0 = es[PPOAF_ST_ACTOR_LOSS], e1 = es[PPOAF_ST_CRITIC_LOSS], e2 = es[PPOAF_ST_ENTROPY], e3 = es[PPOAF_ST_KL];
    const double e4 = es[PPOAF_ST_COUNTER], e5 = es[PPOAF_ST_BAD_RATIO], e6 = es[PPOAF_ST_BAD_VALUE];   // loads, then stores
    es[PPOAF_ST_ACTOR_LOSS] = e0 + double(actor_mean);
    es[PPOAF_ST_CRITIC_LOSS] = e1 + double(critic_mean);
    if (w_ent != 0.f) es[PPOAF_ST_ENTROPY] = e2 + double(float(s_tot[LS_ENTROPY] / nb));
    es[PPOAF_ST_KL] = e3 + double(float(s_tot[LS_KL] / nb));
    es[PPOAF_ST_COUNTER] = e4 + 1.0;
    es[PPOAF_ST_BAD_RATIO] = e5 + s_tot[LS_BAD_RATIO];
    es[PPOAF_ST_BAD_VALUE] = e6 + s_tot[LS_BAD_VALUE];
}

}  // namespace ppoaf
