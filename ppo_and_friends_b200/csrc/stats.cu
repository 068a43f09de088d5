// Running statistics (RunningMeanStd, reference utils/stats.py:9-94) and the normalisers built on
// them (utils/misc.py:84-128; environments/filter_wrappers.py:220-221, 655-657).
//
// Column moments of x[n_rows, dim]: every thread owns one float4 column group and walks down the
// rows (coalesced 128-bit loads, 4 rows in flight), keeping fp32 Welford state; partials are merged
// with Chan's formula in fp64: across threadIdx.y in shared memory, across CTAs by a second kernel
// in which one warp per column tree-merges the CTA partials with shuffles.
#include "internal.h"

namespace ppoaf {

#ifndef PPOAF_STAT_ROWS
#define PPOAF_STAT_ROWS 8
#endif
#ifndef PPOAF_STAT_UNROLL
#define PPOAF_STAT_UNROLL 4
#endif
#ifndef PPOAF_STAT_GRID_MULT
#define PPOAF_STAT_GRID_MULT 32
#endif
constexpr int kStatRowsPerBlock = PPOAF_STAT_ROWS;   // blockDim.y
constexpr int kStatUnroll = PPOAF_STAT_UNROLL;       // rows in flight per thread
constexpr int kMaxFoldWidth = 128;     // narrow rows are folded k-at-a-time up to this many floats

struct FoldPlan {
    int fold;          // rows folded into one super-row (1 = none)
    int width;         // dim * fold (multiple of 4)
    int64_t rows;      // super-rows
    int64_t tail;      // leftover original rows (< fold), handled by the finalize kernel
    int vec;           // width / 4
    int bx;            // blockDim.x (vec rounded up to a warp multiple)
    int grid;
    bool ok;
};

static FoldPlan plan_fold(int64_t n_rows, int32_t dim, const void* p) {
    FoldPlan f{};
    f.ok = false;
    if (reinterpret_cast<uintptr_t>(p) % 16 != 0) return f;
    int fold = 1;
    if (dim < kMaxFoldWidth) {
        fold = kMaxFoldWidth / dim;
        while (fold > 1 && (int64_t(dim) * fold) % 4 != 0) --fold;
    }
    if ((int64_t(dim) * fold) % 4 != 0) return f;
    f.fold = fold;
    f.width = dim * fold;
    f.rows = n_rows / fold;
    f.tail = n_rows - f.rows * fold;
    f.vec = f.width / 4;
    f.bx = (f.vec + 31) / 32 * 32;
    if (f.bx * kStatRowsPerBlock > 1024) return f;  // dim > 1024: generic path
    const int64_t want = ceil_div64(f.rows, int64_t(kStatRowsPerBlock) * kStatUnroll * (fold > 1 ? 2 : 8));
#ifndef PPOAF_STAT_GRID_MULT_M
#define PPOAF_STAT_GRID_MULT_M 4
#endif
    const int64_t cap = int64_t(sm_count()) * PPOAF_STAT_GRID_MULT_M;
    f.grid = int(want < 1 ? 1 : (want > cap ? cap : want));
    f.ok = f.rows > 0;
    return f;
}

__device__ __forceinline__ void welford4(float4 x, float rn, float4& mean, float4& m2) {
    float d;
    d = x.x - mean.x; mean.x = fmaf(d, rn, mean.x); m2.x = fmaf(d, x.x - mean.x, m2.x);
    d = x.y - mean.y; mean.y = fmaf(d, rn, mean.y); m2.y = fmaf(d, x.y - mean.y, m2.y);
    d = x.z - mean.z; mean.z = fmaf(d, rn, mean.z); m2.z = fmaf(d, x.z - mean.z, m2.z);
    d = x.w - mean.w; mean.w = fmaf(d, rn, mean.w); m2.w = fmaf(d, x.w - mean.w, m2.w);
}

// partial[(block * width + col) * 3 + {0,1,2}] = n, mean, M2
// fold > 1 (narrow rows folded `fold` at a time into super-rows of `width` floats): the CTA also merges the fold copies of
// every true column, so it publishes `dim` triples instead of `width` and the finalize kernel has fold x fewer to fold.
// Rows of 388..512 floats run it with 1024 threads, which leaves at most 64 registers a thread.
__global__ void __launch_bounds__(1024)
moments_partial_kernel(const float4* __restrict__ x, int64_t rows, int vec, int dim, int fold,
                       double* __restrict__ partial) {
    extern __shared__ double s_part[];  // [blockDim.y][vec*4][2] mean, m2 ; counts in s_cnt
    __shared__ float s_cnt[kStatRowsPerBlock];
    const int g = threadIdx.x, y = threadIdx.y;
    const int64_t per_block = ceil_div64(rows, gridDim.x);
    const int64_t r0 = int64_t(blockIdx.x) * per_block;
    const int64_t r1 = min(r0 + per_block, rows);
    float4 mean = make_float4(0.f, 0.f, 0.f, 0.f), m2 = mean;
    float n = 0.f;
    if (g < vec) {
        int64_t r = r0 + y;
        const int64_t step = kStatRowsPerBlock;
        for (; r + (kStatUnroll - 1) * step < r1; r += kStatUnroll * step) {
            float4 v[kStatUnroll];
#pragma unroll
            for (int u = 0; u < kStatUnroll; ++u) v[u] = ldg_stream_f4(x + (r + u * step) * vec + g);
#pragma unroll
            for (int u = 0; u < kStatUnroll; ++u) {
                n += 1.f;
                welford4(v[u], __frcp_rn(n), mean, m2);
            }
        }
        for (; r < r1; r += step) {
            const float4 v = ldg_stream_f4(x + r * vec + g);
            n += 1.f;
            welford4(v, __frcp_rn(n), mean, m2);
        }
        double* sp = s_part + (size_t(y) * vec * 4 + size_t(g) * 4) * 2;
        sp[0] = mean.x; sp[1] = m2.x; sp[2] = mean.y; sp[3] = m2.y;
        sp[4] = mean.z; sp[5] = m2.z; sp[6] = mean.w; sp[7] = m2.w;
        if (g == 0) s_cnt[y] = n;
    }
    __syncthreads();
    // merge the blockDim.y row-lanes per column, fp64
    const int width = vec * 4;
    Moments* s_fold = reinterpret_cast<Moments*>(s_part + size_t(kStatRowsPerBlock) * width * 2);   // only allocated when fold > 1
    for (int c = threadIdx.y * blockDim.x + threadIdx.x; c < width; c += blockDim.x * blockDim.y) {
        Moments acc{0.0, 0.0, 0.0};
        for (int yy = 0; yy < kStatRowsPerBlock; ++yy) {
            const double* sp = s_part + (size_t(yy) * width + c) * 2;
            Moments m{double(s_cnt[yy]), sp[0], sp[1]};
            acc = merge_moments(acc, m);
        }
        if (fold > 1) {
            s_fold[c] = acc;                                   // width <= kMaxFoldWidth whenever fold > 1
        } else {
            double* out = partial + (size_t(blockIdx.x) * width + c) * 3;
            out[0] = acc.n; out[1] = acc.mean; out[2] = acc.m2;
        }
    }
    if (fold > 1) {                                            // column c = j * dim + col: tree over the fold index j
        const int tid = threadIdx.y * blockDim.x + threadIdx.x;
        int p2 = 1;
        while (p2 < fold) p2 <<= 1;
        for (int stride = p2 >> 1; stride >= 1; stride >>= 1) {
            __syncthreads();
            for (int c = tid; c < stride * dim; c += blockDim.x * blockDim.y) {
                const int j = c / dim;
                if (j + stride < fold) s_fold[c] = merge_moments(s_fold[c], s_fold[c + stride * dim]);
            }
        }
        __syncthreads();
        for (int col = tid; col < dim; col += blockDim.x * blockDim.y) {
            double* out = partial + (size_t(blockIdx.x) * dim + col) * 3;
            out[0] = s_fold[col].n; out[1] = s_fold[col].mean; out[2] = s_fold[col].m2;
        }
    }
}

// One CTA per TRUE column: threads stride over the (CTA, fold) partials, then a shuffle tree merge inside
// each warp and a fixed-order merge of the warps (Chan), so the result is deterministic.
constexpr int kFinThreads = 128;       // wide rows: few partials per column
constexpr int kFinThreadsMax = 1024;   // folded narrow rows (dim = 1: n_blocks x 128 partials in ONE column): one full CTA
__global__ void __launch_bounds__(kFinThreadsMax)
moments_finalize_kernel(const double* __restrict__ partial, int n_blocks, int width, int dim, int fold,
                        const float* __restrict__ tail_rows, int64_t tail, double* __restrict__ triple_out) {
    __shared__ Moments s_w[kFinThreadsMax / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
    const int col = blockIdx.x;
    Moments acc{0.0, 0.0, 0.0};
    const int items = n_blocks * fold;
    for (int it = threadIdx.x; it < items; it += blockDim.x) {
        const int b = it / fold, j = it - b * fold;
        const double* p = partial + (size_t(b) * width + size_t(j) * dim + col) * 3;
        Moments m{p[0], p[1], p[2]};
        acc = merge_moments(acc, m);
    }
    for (int64_t t = threadIdx.x; t < tail; t += blockDim.x) {
        Moments m{1.0, double(tail_rows[t * dim + col]), 0.0};
        acc = merge_moments(acc, m);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const Moments other = shfl_xor_moments(acc, o);
        // merge in a fixed (lower lane first) order so both partners compute the same bits
        acc = (lane & o) ? merge_moments(other, acc) : merge_moments(acc, other);
    }
    if (lane == 0) s_w[warp] = acc;
    __syncthreads();
    if (warp == 0) {                       // the warp results meet in a second fixed-order shuffle tree
        Moments t = lane < n_warps ? s_w[lane] : Moments{0.0, 0.0, 0.0};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const Moments other = shfl_xor_moments(t, o);
            t = (lane & o) ? merge_moments(other, t) : merge_moments(t, other);
        }
        if (lane == 0) {
            triple_out[col] = t.mean;
            triple_out[dim + col] = t.m2;
            if (col == 0) triple_out[2 * dim] = t.n;
        }
    }
}

// Generic fallback (unaligned base / odd widths): one warp per column striding over rows.
__global__ void moments_generic_kernel(const float* __restrict__ x, int64_t n_rows, int dim,
                                       double* __restrict__ triple_out) {
    const int lane = threadIdx.x & 31;
    const int col = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (col >= dim) return;
    Moments acc{0.0, 0.0, 0.0};
    for (int64_t r = lane; r < n_rows; r += 32) {
        const double v = double(x[r * dim + col]);
        acc.n += 1.0;
        const double d = v - acc.mean;
        acc.mean += d / acc.n;
        acc.m2 += d * (v - acc.mean);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const Moments other = shfl_xor_moments(acc, o);
        acc = (lane & o) ? merge_moments(other, acc) : merge_moments(acc, other);
    }
    if (lane == 0) {
        triple_out[col] = acc.mean;
        triple_out[dim + col] = acc.m2;
        if (col == 0) triple_out[2 * dim] = acc.n;
    }
}

// state = mean[dim] | var[dim] | count ; triples = n_triples x (mean[dim] | M2[dim] | n)
__global__ void stats_merge_kernel(double* __restrict__ state, const double* __restrict__ triples, int n_triples,
                                   int dim) {
    const double count = state[2 * dim];
    double n_tot = 0.0;
    for (int t = 0; t < n_triples; ++t) n_tot += triples[size_t(t) * (2 * dim + 1) + 2 * dim];
    for (int c = threadIdx.x; c < dim; c += blockDim.x) {
        Moments pool{0.0, 0.0, 0.0};
        for (int t = 0; t < n_triples; ++t) {
            const double* tr = triples + size_t(t) * (2 * dim + 1);
            Moments m{tr[2 * dim], tr[c], tr[dim + c]};
            pool = merge_moments(pool, m);
        }
        if (pool.n > 0.0) {
            // RunningMeanStd._integrate_batch_data (utils/stats.py:73-94)
            const double bmean = pool.mean, bvar = pool.m2 / pool.n, bn = pool.n;
            const double mean = state[c], var = state[dim + c];
            const double delta = bmean - mean;
            const double tot = count + bn;
            state[c] = mean + delta * (bn / tot);
            const double m_2 = var * count + bvar * bn + delta * delta * count * bn / (count + bn);
            state[dim + c] = m_2 / (count + bn);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) state[2 * dim] = count + n_tot;
}

template <bool kDenorm>
__global__ void normalize_vec_kernel(const float4* __restrict__ x, float4* __restrict__ y, int64_t rows, int vec,
                                     int dim, const double* __restrict__ state, float eps, float lo, float hi) {
    const int g = threadIdx.x;
    if (g >= vec) return;
    float mu[4], sc[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int c = (g * 4 + k) % dim;
        mu[k] = float(state[c]);
        const float sd = sqrtf(float(state[dim + c]) + eps);
        sc[k] = kDenorm ? sd : 1.0f / sd;
    }
    const bool clip = lo < hi;
    const int64_t per_block = ceil_div64(rows, gridDim.x);
    const int64_t r0 = int64_t(blockIdx.x) * per_block;
    const int64_t r1 = min(r0 + per_block, rows);
    const int64_t step = blockDim.y;
    auto apply = [&](float4 v) {
        float o[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            o[k] = kDenorm ? fmaf(o[k], sc[k], mu[k]) : (o[k] - mu[k]) * sc[k];
            if (clip) o[k] = fminf(fmaxf(o[k], lo), hi);
        }
        return make_float4(o[0], o[1], o[2], o[3]);
    };
    int64_t r = r0 + threadIdx.y;
    for (; r + (kStatUnroll - 1) * step < r1; r += kStatUnroll * step) {
        float4 v[kStatUnroll];
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) v[u] = ldg_stream_f4(x + (r + u * step) * vec + g);
#pragma unroll
        for (int u = 0; u < kStatUnroll; ++u) stg_stream_f4(y + (r + u * step) * vec + g, apply(v[u]));
    }
    for (; r < r1; r += step) stg_stream_f4(y + r * vec + g, apply(ldg_stream_f4(x + r * vec + g)));
}

template <bool kDenorm>
__global__ void normalize_scalar_kernel(const float* __restrict__ x, float* __restrict__ y, int64_t total, int dim,
                                        const double* __restrict__ state, float eps, float lo, float hi) {
    const bool clip = lo < hi;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int c = int(i % dim);
        const float mu = float(state[c]);
        const float sd = sqrtf(float(state[dim + c]) + eps);
        float o = kDenorm ? fmaf(x[i], sd, mu) : (x[i] - mu) / sd;
        if (clip) o = fminf(fmaxf(o, lo), hi);
        y[i] = o;
    }
}

// ---- per-epoch minibatch tables ------------------------------------------------------------------
__global__ void epoch_prepare_kernel(const int64_t* __restrict__ perm, const float* __restrict__ adv,
                                     const float* __restrict__ rtg, int64_t n, int batch_size,
                                     float* __restrict__ mb_adv_stats, double* __restrict__ mb_val_triples) {
    __shared__ Moments s_a[32], s_r[32];
    const int k = blockIdx.x;
    const int64_t lo = int64_t(k) * batch_size;
    const int cnt = int(min(int64_t(batch_size), n - lo));
    Moments a{0.0, 0.0, 0.0}, r{0.0, 0.0, 0.0};
    for (int i = threadIdx.x; i < cnt; i += blockDim.x) {
        const int64_t j = perm[lo + i];
        const double av = double(adv[j]), rv = double(rtg[j]);
        a.n += 1.0; double d = av - a.mean; a.mean += d / a.n; a.m2 += d * (av - a.mean);
        r.n += 1.0; d = rv - r.mean; r.mean += d / r.n; r.m2 += d * (rv - r.mean);
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const Moments oa = shfl_xor_moments(a, o), orr = shfl_xor_moments(r, o);
        a = (lane & o) ? merge_moments(oa, a) : merge_moments(a, oa);
        r = (lane & o) ? merge_moments(orr, r) : merge_moments(r, orr);
    }
    if (lane == 0) { s_a[warp] = a; s_r[warp] = r; }
    __syncthreads();
    if (threadIdx.x == 0) {
        Moments ta = s_a[0], tr = s_r[0];
        for (int w = 1; w < nw; ++w) { ta = merge_moments(ta, s_a[w]); tr = merge_moments(tr, s_r[w]); }
        // torch.std is the unbiased (N-1) estimator (ppo.py:2326); one row gives nan like torch
        const float mean = float(ta.mean);
        const float sd = float(sqrt(ta.m2 / (ta.n - 1.0)));
        mb_adv_stats[2 * k] = mean;
        mb_adv_stats[2 * k + 1] = sd + 1e-8f;
        mb_val_triples[3 * k] = tr.mean;
        mb_val_triples[3 * k + 1] = tr.m2;
        mb_val_triples[3 * k + 2] = tr.n;
    }
}

__global__ void value_stats_sequence_kernel(double* __restrict__ state, const double* __restrict__ triples,
                                            int n_ranks, int n_mb, float eps, float* __restrict__ mb_val_stats) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double mean = state[0], var = state[1], count = state[2];
    for (int k = 0; k < n_mb; ++k) {
        Moments pool{0.0, 0.0, 0.0};
        for (int r = 0; r < n_ranks; ++r) {
            const double* t = triples + (size_t(r) * n_mb + k) * 3;
            Moments m{t[2], t[0], t[1]};
            pool = merge_moments(pool, m);
        }
        if (pool.n > 0.0) {
            const double bmean = pool.mean, bvar = pool.m2 / pool.n, bn = pool.n;
            const double delta = bmean - mean, tot = count + bn;
            const double m_2 = var * count + bvar * bn + delta * delta * count * bn / (count + bn);
            mean = mean + delta * (bn / tot);
            var = m_2 / (count + bn);
            count = tot;
        }
        mb_val_stats[2 * k] = float(mean);
        mb_val_stats[2 * k + 1] = sqrtf(float(var) + eps);
    }
    state[0] = mean; state[1] = var; state[2] = count;
}

// ---- reward normaliser, one environment step (reference environments/filter_wrappers.py:393-425, SURVEY Q9) ----
// The reference walks the E environments of a rank IN ORDER: running_reward[e] = running_reward[e] * gamma + r[e], and
// after EVERY single-element change it feeds the WHOLE (partially updated) vector to RunningMeanStd.update — E statistic
// updates per step.  The moments of a vector in which one element changed follow from the previous ones in O(1) (fp64),
// so one thread produces the E batch triples (mean, M2, n = E) of a step; ppoaf_value_stats_sequence then pools them over
// ranks and integrates them in (e, rank) order, exactly like the reference's allgather + concatenate inside the loop.
__global__ void reward_norm_triples_kernel(const float* __restrict__ rewards, const uint8_t* __restrict__ dones,
                                           double* __restrict__ running_reward, int E, double gamma,
                                           double* __restrict__ triples) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    double mean = 0.0;
    for (int e = 0; e < E; ++e) mean += running_reward[e];
    mean /= double(E);
    double m2 = 0.0;
    for (int e = 0; e < E; ++e) { const double d = running_reward[e] - mean; m2 += d * d; }
    for (int e = 0; e < E; ++e) {
        const double old = running_reward[e];
        // rounded product then rounded sum, as the reference's numpy does: a contracted fma would drift from it
        const double nw = __dadd_rn(__dmul_rn(old, gamma), double(rewards[e]));
        running_reward[e] = nw;
        const double new_mean = mean + (nw - old) / double(E);
        m2 += (nw - old) * ((nw - new_mean) + (old - mean));
        if (m2 < 0.0) m2 = 0.0;
        mean = new_mean;
        triples[3 * e] = mean; triples[3 * e + 1] = m2; triples[3 * e + 2] = double(E);
    }
    for (int e = 0; e < E; ++e)
        if (dones[e]) running_reward[e] = 0.0;               // filter_wrappers.py:420-425
}

// y = clip(r / sqrt(var + eps), lo, hi)  (filter_wrappers.py:466-476 followed by RewardClipper :700-719); lo >= hi: no clip
__global__ void reward_scale_clip_kernel(const float* __restrict__ r, const double* __restrict__ state, float eps, float lo,
                                         float hi, float* __restrict__ y, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double sd = sqrt(state[1] + double(eps));
    float v = float(double(r[i]) / sd);
    if (lo < hi) v = fminf(fmaxf(v, lo), hi);
    y[i] = v;
}

// The widest vectorised moments plan is fold = 1 with blockDim.x * kStatRowsPerBlock = 1024 threads, i.e. rows of 512
// floats, whose per-row-lane (mean, M2) partials take 64 KB of dynamic shared memory: more than the 48 KB a kernel may
// use without opting in.
constexpr int kMaxVecWidth = 4 * 1024 / kStatRowsPerBlock;
constexpr size_t kMomentsSmemMax = size_t(kStatRowsPerBlock) * kMaxVecWidth * 2 * sizeof(double);
static_assert(size_t(kStatRowsPerBlock) * kMaxFoldWidth * 2 * sizeof(double) + kMaxFoldWidth * sizeof(Moments) <=
              kMomentsSmemMax, "folded plans need more shared memory than the widest unfolded one");

// Called from ppoaf_runtime_init (so that the attribute call normally happens before any stream capture) and, for callers
// of the C ABI that never initialise the runtime, lazily by the first ppoaf_batch_moments.
static bool g_stats_configured = false;
void configure_stats_kernels() {
    g_stats_configured = true;
    cudaFuncSetAttribute(moments_partial_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kMomentsSmemMax));
}

}  // namespace ppoaf

using namespace ppoaf;

extern "C" int ppoaf_reward_norm_triples(const float* rewards, const uint8_t* dones, double* running_reward, int32_t n_envs,
                                         double gamma, double* triples_out, void* stream) {
    PPOAF_CHECK_ARG(n_envs > 0 && rewards && dones && running_reward && triples_out, "ppoaf_reward_norm_triples: bad arguments");
    reward_norm_triples_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rewards, dones, running_reward, n_envs, gamma, triples_out);
    PPOAF_CHECK_LAUNCH("ppoaf_reward_norm_triples");
    return 0;
}

extern "C" int ppoaf_reward_scale_clip(const float* rewards, const double* state, float eps, float lo, float hi, float* out,
                                       int32_t n, void* stream) {
    PPOAF_CHECK_ARG(n >= 0, "ppoaf_reward_scale_clip: n < 0");
    if (n == 0) return 0;
    reward_scale_clip_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(rewards, state, eps, lo, hi, out, n);
    PPOAF_CHECK_LAUNCH("ppoaf_reward_scale_clip");
    return 0;
}

extern "C" size_t ppoaf_moments_workspace_bytes(int64_t n_rows, int32_t dim) {
    if (n_rows <= 0 || dim <= 0) return 64;
    // upper bound independent of pointer alignment: grid <= 4*SMs, width <= max(dim, kMaxFoldWidth)
    const size_t width = size_t(dim < kMaxFoldWidth ? kMaxFoldWidth : dim);
    return size_t(sm_count()) * 4 * width * 3 * sizeof(double) + 64;
}

extern "C" int ppoaf_batch_moments(const float* x, int64_t n_rows, int32_t dim, double* triple_out, void* workspace,
                                   size_t workspace_bytes, void* stream) {
    PPOAF_CHECK_ARG(n_rows > 0 && dim > 0, "ppoaf_batch_moments: needs n_rows > 0 and dim > 0");
    cudaStream_t s = (cudaStream_t)stream;
    const FoldPlan f = plan_fold(n_rows, dim, x);
    const int warps_per_block = 8;
    const int fin_blocks = (dim + warps_per_block - 1) / warps_per_block;
    if (!f.ok) {
        moments_generic_kernel<<<fin_blocks, warps_per_block * 32, 0, s>>>(x, n_rows, dim, triple_out);
        PPOAF_CHECK_LAUNCH("ppoaf_batch_moments(generic)");
        return 0;
    }
    PPOAF_CHECK_ARG(workspace_bytes >= size_t(f.grid) * f.width * 3 * sizeof(double),
                    "ppoaf_batch_moments: workspace too small");
    PPOAF_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 8 == 0, "ppoaf_batch_moments: workspace alignment");
    double* partial = reinterpret_cast<double*>(workspace);
    if (!g_stats_configured) configure_stats_kernels();
    const dim3 block(f.bx, kStatRowsPerBlock);
    const size_t smem = size_t(kStatRowsPerBlock) * f.width * 2 * sizeof(double) + (f.fold > 1 ? size_t(f.width) * sizeof(Moments) : 0);
    moments_partial_kernel<<<f.grid, block, smem, s>>>(reinterpret_cast<const float4*>(x), f.rows, f.vec, dim, f.fold, partial);
    PPOAF_CHECK_LAUNCH("ppoaf_batch_moments(partial)");
    // (folded inputs arrive already merged over the fold index: one triple per CTA and true column)
    const int fin_threads = f.grid >= 2048 ? kFinThreadsMax : kFinThreads;
    moments_finalize_kernel<<<dim, fin_threads, 0, s>>>(
        partial, f.grid, f.fold > 1 ? dim : f.width, dim, 1, x + f.rows * f.fold * int64_t(dim), f.tail, triple_out);
    PPOAF_CHECK_LAUNCH("ppoaf_batch_moments(finalize)");
    return 0;
}

extern "C" int ppoaf_stats_merge(double* state, const double* triples, int32_t n_triples, int32_t dim, void* stream) {
    PPOAF_CHECK_ARG(n_triples >= 0 && dim > 0, "ppoaf_stats_merge: bad sizes");
    if (n_triples == 0) return 0;
    stats_merge_kernel<<<1, 256, 0, (cudaStream_t)stream>>>(state, triples, n_triples, dim);
    PPOAF_CHECK_LAUNCH("ppoaf_stats_merge");
    return 0;
}

template <bool kDenorm>
static int launch_normalize(const float* x, int64_t n_rows, int32_t dim, const double* state, float eps, float lo,
                            float hi, float* y, cudaStream_t s) {
    if (n_rows == 0) return 0;
    FoldPlan f = plan_fold(n_rows, dim, x);
    if (f.ok && reinterpret_cast<uintptr_t>(y) % 16 != 0) f.ok = false;
    if (f.ok) {
        const int64_t want = ceil_div64(f.rows, int64_t(kStatRowsPerBlock) * kStatUnroll * 4);
        const int64_t cap = int64_t(sm_count()) * PPOAF_STAT_GRID_MULT;
        const int grid = int(want < 1 ? 1 : (want > cap ? cap : want));
        normalize_vec_kernel<kDenorm><<<grid, dim3(f.bx, kStatRowsPerBlock), 0, s>>>(
            reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(y), f.rows, f.vec, dim, state, eps, lo, hi);
        PPOAF_CHECK_LAUNCH("ppoaf_normalize(vec)");
        if (f.tail > 0) {
            const int64_t off = f.rows * f.fold * int64_t(dim);
            normalize_scalar_kernel<kDenorm><<<1, 256, 0, s>>>(x + off, y + off, f.tail * dim, dim, state, eps, lo, hi);
            PPOAF_CHECK_LAUNCH("ppoaf_normalize(tail)");
        }
        return 0;
    }
    const int64_t total = n_rows * dim;
    int64_t blocks = ceil_div64(total, 256);
    const int64_t cap = int64_t(sm_count()) * 8;
    if (blocks > cap) blocks = cap;
    normalize_scalar_kernel<kDenorm><<<(unsigned)blocks, 256, 0, s>>>(x, y, total, dim, state, eps, lo, hi);
    PPOAF_CHECK_LAUNCH("ppoaf_normalize(scalar)");
    return 0;
}

extern "C" int ppoaf_normalize_clip(const float* x, int64_t n_rows, int32_t dim, const double* state, float eps,
                                    float lo, float hi, float* y, void* stream) {
    PPOAF_CHECK_ARG(n_rows >= 0 && dim > 0, "ppoaf_normalize_clip: bad sizes");
    return launch_normalize<false>(x, n_rows, dim, state, eps, lo, hi, y, (cudaStream_t)stream);
}

extern "C" int ppoaf_denormalize(const float* x, int64_t n_rows, int32_t dim, const double* state, float eps,
                                 float* y, void* stream) {
    PPOAF_CHECK_ARG(n_rows >= 0 && dim > 0, "ppoaf_denormalize: bad sizes");
    return launch_normalize<true>(x, n_rows, dim, state, eps, 1.f, -1.f, y, (cudaStream_t)stream);
}

extern "C" int ppoaf_epoch_prepare(const int64_t* perm, const float* advantages, const float* rewards_to_go,
                                   int64_t n_flat, int32_t batch_size, float* mb_adv_stats, double* mb_val_triples,
                                   void* stream) {
    PPOAF_CHECK_ARG(n_flat > 0 && batch_size > 0, "ppoaf_epoch_prepare: bad sizes");
    const int n_mb = int(ceil_div64(n_flat, batch_size));
    const int threads = batch_size >= 256 ? 256 : (batch_size >= 64 ? 64 : 32);
    epoch_prepare_kernel<<<n_mb, threads, 0, (cudaStream_t)stream>>>(perm, advantages, rewards_to_go, n_flat,
                                                                     batch_size, mb_adv_stats, mb_val_triples);
    PPOAF_CHECK_LAUNCH("ppoaf_epoch_prepare");
    return 0;
}

extern "C" int ppoaf_value_stats_sequence(double* state, const double* mb_val_triples, int32_t n_ranks, int32_t n_mb,
                                          float eps, float* mb_val_stats, void* stream) {
    PPOAF_CHECK_ARG(n_ranks > 0 && n_mb > 0, "ppoaf_value_stats_sequence: bad sizes");
    value_stats_sequence_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(state, mb_val_triples, n_ranks, n_mb, eps,
                                                                     mb_val_stats);
    PPOAF_CHECK_LAUNCH("ppoaf_value_stats_sequence");
    return 0;
}
