// Gradient averaging scale, per-network clip_grad_norm_ and Adam over the flat [actor | critic]
// buffers (reference policies/ppo_policy.py:1032-1055, utils/mpi_utils.py:89-111; arithmetic of
// torch nn/utils/clip_grad.py and optim/adam.py `_single_tensor_adam`, eps = 1e-5 set by the
// reference), as ONE element-wise launch: the per-network sums of squares arrive as fp64 slots
// written by the backward-w GEMM epilogues (single rank) or by a norm pass over the all-reduced
// buffer (R > 1); every CTA folds the slots in a fixed order, derives this step's scalars (clip
// coefficients, bias corrections from the device-side step counter) and updates its slice.  The last
// CTA to finish advances the step / minibatch counters.  HBM traffic: 16 B read + 12 B written per
// parameter.
#include "internal.h"

namespace ppoaf {

constexpr int kOptThreads = 256;
constexpr int kAdamThreads = 1024;      // adam_update_kernel: 148 x 1024 threads, two float4 slots each, cover 1.2 M parameters in one pass
constexpr int kAdamSlots = 2;

// Norm pass for the multi-rank path: fixed-order fp64 partials per CTA, no atomics.
__global__ void __launch_bounds__(kOptThreads)
grad_sumsq_kernel(const float* __restrict__ grads, int64_t n_actor, int64_t n_total, double* __restrict__ part_a,
                  double* __restrict__ part_c) {
    __shared__ double s_scr[32];
    const float4* g4 = reinterpret_cast<const float4*>(grads);
    const int64_t nv = n_total / 4, na = n_actor / 4;
    double sa = 0.0, sc = 0.0;
    for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < nv; i += int64_t(gridDim.x) * blockDim.x) {
        const float4 x = g4[i];
        const float q = fmaf(x.x, x.x, fmaf(x.y, x.y, fmaf(x.z, x.z, x.w * x.w)));
        if (i < na) sa += double(q); else sc += double(q);
    }
    sa = block_sum(sa, s_scr);
    sc = block_sum(sc, s_scr);
    if (threadIdx.x == 0) { part_a[blockIdx.x] = sa; part_c[blockIdx.x] = sc; }
}

struct AdamScalars { float neg_step_size, bc2_sqrt, w1, beta2, w2, eps, inv_world; };
__device__ __forceinline__ void adam_vec(float4& pq, const float4& gq, float4& mq, float4& vq, float coef, const AdamScalars& c) {
    float g[4] = {gq.x, gq.y, gq.z, gq.w}, p[4] = {pq.x, pq.y, pq.z, pq.w};
    float mm[4] = {mq.x, mq.y, mq.z, mq.w}, vv[4] = {vq.x, vq.y, vq.z, vq.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        // explicit _rn intrinsics: same operation order as torch's CPU kernels, no FMA contraction
        const float gk = __fmul_rn(__fmul_rn(g[k], c.inv_world), coef);
        mm[k] = __fadd_rn(mm[k], __fmul_rn(c.w1, __fsub_rn(gk, mm[k])));                   // lerp_(g, 1-b1)
        vv[k] = __fadd_rn(__fmul_rn(vv[k], c.beta2), __fmul_rn(__fmul_rn(c.w2, gk), gk));   // mul_ ; addcmul_
        // sqrt and the two divisions use the approximate units (<= 2 ulp each): the IEEE sequences were ~75 of the ~100
        // instructions per parameter and made the kernel latency-bound (ncu, round 2); the effect on a parameter is
        // ~lr * 5e-7 relative to the update, far inside the 2e-6 agreement with torch.optim.Adam that the tests check
        float sq;
        asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(vv[k]));
        const float denom = __fadd_rn(__fdividef(sq, c.bc2_sqrt), c.eps);
        p[k] = __fadd_rn(p[k], __fdividef(__fmul_rn(c.neg_step_size, mm[k]), denom));       // addcdiv_
    }
    pq = make_float4(p[0], p[1], p[2], p[3]);
    mq = make_float4(mm[0], mm[1], mm[2], mm[3]);
    vq = make_float4(vv[0], vv[1], vv[2], vv[3]);
}

__global__ void __launch_bounds__(kAdamThreads)
adam_update_kernel(float* __restrict__ params, const float* __restrict__ grads, float* __restrict__ m,
                   float* __restrict__ v, int64_t n_actor, int64_t n_total, const double* __restrict__ sq_a,
                   int n_sq_a, const double* __restrict__ sq_c, int n_sq_c, const double* __restrict__ hp,
                   int64_t* __restrict__ adam_step, int32_t* __restrict__ mb_cursor, unsigned int* __restrict__ ticket) {
    __shared__ double s_scr[32];
    __shared__ double s_pw[2];
    __shared__ float s_coef[2];
    double* pw = reinterpret_cast<double*>(ticket + 2);   // cached (t, beta1, beta2, beta1^t, beta2^t)
    const int64_t nv = n_total / 4, na = n_actor / 4;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    const int64_t i0 = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
    float4* p4 = reinterpret_cast<float4*>(params);
    const float4* g4 = reinterpret_cast<const float4*>(grads);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);

    // ---- the first kAdamSlots float4 slots of every thread are in flight while the scalars are derived; the
    // parameters and moments (only ever written by this kernel) are fetched before the dependency wait ----
    float4 G[kAdamSlots], P[kAdamSlots], M[kAdamSlots], V[kAdamSlots];
#pragma unroll
    for (int k = 0; k < kAdamSlots; ++k) {
        const int64_t i = i0 + k * stride;
        if (i < nv) { P[k] = p4[i]; M[k] = m4[i]; V[k] = v4[i]; }
    }
    pdl_wait();
    pdl_trigger();
#pragma unroll
    for (int k = 0; k < kAdamSlots; ++k) {
        const int64_t i = i0 + k * stride;
        if (i < nv) G[k] = g4[i];
    }

    // ---- fold the sum-of-squares slots (same order in every CTA -> identical scalars everywhere) ----
    double ta = 0.0, tc = 0.0;
    for (int k = threadIdx.x; k < n_sq_a; k += blockDim.x) ta += sq_a[k];
    for (int k = threadIdx.x; k < n_sq_c; k += blockDim.x) tc += sq_c[k];
    ta = block_sum(ta, s_scr);
    tc = block_sum(tc, s_scr);
    const float inv_world = float(hp[PPOAF_HP_INV_WORLD]);
    if (threadIdx.x == 0) {
        const float max_norm = float(hp[PPOAF_HP_GRAD_CLIP]);
        // the slots hold sums over the SUMMED gradients; the averaged gradient is inv_world times that
        s_coef[0] = clip_coef(max_norm, ta, double(inv_world));
        s_coef[1] = clip_coef(max_norm, tc, double(inv_world));
    }
    const int64_t t = *adam_step + 1;
    __shared__ float s_f[6];
    if (threadIdx.x == 0) {
        const double b1d = hp[PPOAF_HP_BETA1], b2d = hp[PPOAF_HP_BETA2];
        double p1, p2;
        beta_powers(pw, t, b1d, b2d, p1, p2);
        s_pw[0] = p1; s_pw[1] = p2;
        const double bc1 = 1.0 - p1;
        const double bc2 = 1.0 - p2;
        s_f[0] = float(-(hp[PPOAF_HP_LR] / bc1));     // -step_size = -lr / (1 - beta1^t)
        s_f[1] = float(sqrt(bc2));                    // sqrt(1 - beta2^t)
        s_f[2] = float(1.0 - b1d);
        s_f[3] = float(b2d);
        s_f[4] = float(1.0 - b2d);
        s_f[5] = float(hp[PPOAF_HP_ADAM_EPS]);
    }
    __syncthreads();
    const AdamScalars c{s_f[0], s_f[1], s_f[2], s_f[3], s_f[4], s_f[5], inv_world};
    const float coef_a = s_coef[0], coef_c = s_coef[1];

#pragma unroll
    for (int k = 0; k < kAdamSlots; ++k) {
        const int64_t i = i0 + k * stride;
        if (i < nv) {
            adam_vec(P[k], G[k], M[k], V[k], i < na ? coef_a : coef_c, c);
            p4[i] = P[k]; m4[i] = M[k]; v4[i] = V[k];
        }
    }
    for (int64_t i = i0 + kAdamSlots * stride; i < nv; i += stride) {      // networks beyond 1.2 M parameters
        const float4 gq = g4[i];
        float4 pq = p4[i], mq = m4[i], vq = v4[i];
        adam_vec(pq, gq, mq, vq, i < na ? coef_a : coef_c, c);
        p4[i] = pq; m4[i] = mq; v4[i] = vq;
    }
    // ---- the last CTA to finish advances the counters (every CTA has read adam_step by then) ----
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(ticket, 1u) == gridDim.x - 1) {
            *adam_step = t;
            if (mb_cursor) *mb_cursor += 1;
            store_beta_powers(pw, t, hp[PPOAF_HP_BETA1], hp[PPOAF_HP_BETA2], s_pw[0], s_pw[1]);
            *ticket = 0u;
        }
    }
}

__global__ void advance_cursor_kernel(int32_t* mb_cursor) { *mb_cursor += 1; }

static int opt_grid(int64_t n_total) {
    int64_t b = ceil_div64(n_total / 4, kOptThreads);
    const int64_t cap = int64_t(sm_count());
    return int(b < 1 ? 1 : (b > cap ? cap : b));
}

constexpr size_t kTicketBytes = 256;    // ticket word, one spare word, the beta-power cache
static_assert(2 * sizeof(unsigned int) + kBetaCacheDoubles * sizeof(double) <= kTicketBytes,
              "the beta-power cache must fit the ticket region");
size_t optim_workspace_bytes() {
    return align_up(size_t(sm_count()) * 2 * sizeof(double), 256) + kTicketBytes;  // norm-pass partials | ticket region
}

int launch_clip_adam(float* params, const float* grads, float* m, float* v, int64_t* adam_step, int32_t* mb_cursor,
                     const double* hparams, int64_t n_actor, int64_t n_critic, const double* sq_a, int n_sq_a,
                     const double* sq_c, int n_sq_c, void* workspace, cudaStream_t s, bool chained) {
    PPOAF_CHECK_ARG(n_actor % 4 == 0 && n_critic % 4 == 0, "clip_adam: segment sizes must be multiples of 4 floats");
    PPOAF_CHECK_ARG((reinterpret_cast<uintptr_t>(params) | reinterpret_cast<uintptr_t>(grads) |
                     reinterpret_cast<uintptr_t>(m) | reinterpret_cast<uintptr_t>(v)) % 16 == 0,
                    "clip_adam: buffers must be 16-byte aligned");
    const int64_t n_total = n_actor + n_critic;
    const int grid = opt_grid(n_total);
    double* partials = reinterpret_cast<double*>(workspace);
    unsigned int* ticket = reinterpret_cast<unsigned int*>(
        reinterpret_cast<char*>(workspace) + align_up(size_t(sm_count()) * 2 * sizeof(double), 256));
    if (sq_a == nullptr || sq_c == nullptr) {
        grad_sumsq_kernel<<<grid, kOptThreads, 0, s>>>(grads, n_actor, n_total, partials, partials + grid);
        PPOAF_CHECK_LAUNCH("grad_sumsq_kernel");
        sq_a = partials; sq_c = partials + grid;
        n_sq_a = n_sq_c = grid;
    }
    int64_t agrid = ceil_div64(n_total / 4, kAdamThreads);
    agrid = agrid < 1 ? 1 : (agrid > sm_count() ? sm_count() : agrid);
    // chained: the launch before this one is the last backward GEMM of the step, which never writes params / m / v,
    // so the kernel may fetch them before its dependency wait.  Stand-alone calls keep plain stream order.
    if (chained)
        launch_chain(adam_update_kernel, dim3(int(agrid)), dim3(kAdamThreads), 0, s, params, grads, m, v, n_actor, n_total,
                     sq_a, n_sq_a, sq_c, n_sq_c, hparams, adam_step, mb_cursor, ticket);
    else
        adam_update_kernel<<<int(agrid), kAdamThreads, 0, s>>>(params, grads, m, v, n_actor, n_total, sq_a, n_sq_a, sq_c,
                                                              n_sq_c, hparams, adam_step, mb_cursor, ticket);
    PPOAF_CHECK_LAUNCH("adam_update_kernel");
    return 0;
}

int launch_advance_cursor(int32_t* mb_cursor, cudaStream_t s) {
    advance_cursor_kernel<<<1, 1, 0, s>>>(mb_cursor);
    PPOAF_CHECK_LAUNCH("advance_cursor_kernel");
    return 0;
}

}  // namespace ppoaf

using namespace ppoaf;

extern "C" int ppoaf_clip_adam_step(float* params, const float* grads, float* adam_m, float* adam_v,
                                    int64_t* adam_step, const double* hparams, int64_t n_actor, int64_t n_critic,
                                    void* workspace, size_t workspace_bytes, void* stream) {
    PPOAF_CHECK_ARG(workspace_bytes >= optim_workspace_bytes(), "ppoaf_clip_adam_step: workspace too small");
    PPOAF_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 16 == 0, "ppoaf_clip_adam_step: workspace alignment");
    return launch_clip_adam(params, grads, adam_m, adam_v, adam_step, nullptr, hparams, n_actor, n_critic, nullptr, 0,
                            nullptr, 0, workspace, (cudaStream_t)stream, /*chained=*/false);
}
