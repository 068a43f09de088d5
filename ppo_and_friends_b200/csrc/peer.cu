// Gradient all-reduce over NVLink peer memory FUSED with the gradient-norm clip and Adam
// (replaces: mpi_avg_gradients utils/mpi_utils.py:89-111 + clip_grad_norm_ + Adam.step,
// policies/ppo_policy.py:1032-1055; on the NCCL path that is all-reduce + norm pass + Adam = 3 launches).
//
// Every rank runs this kernel on its own GPU at the same point of the step.  Each rank owns a receive buffer
// [2 step parities][R source ranks][P] mapped into every peer (CUDA IPC over NVSwitch); the backward kernels of
// rank r PUSH every gradient element into slot [parity][r] of every rank's buffer while they run
// (ppoaf_update_bufs.mirror_delta), so by the time this kernel starts the gradients have already crossed NVLink:
//   1. cross-GPU barrier: each rank publishes "my gradients for step t have been written everywhere" by writing t
//      into flag[my_rank] of EVERY peer (st.release.sys over NVLink) and spins on its LOCAL flags until all R
//      ranks have published t;
//   2. one-shot reduce: every thread sums its float4 slots over the R LOCAL slots in rank order (so every rank
//      gets bit-identical sums), keeps them in registers, and accumulates per-network sums of squares;
//   3. local grid barrier (all CTAs are co-resident: grid <= #SMs), fixed-order fold of the CTA partials;
//   4. clip coefficient, bias corrections, Adam on the register-held gradient -> params, m, v (local).
// Because the buffers alternate with step parity, a buffer is rewritten only two steps later, after every
// peer has passed barrier 1 of the step in between — no second cross-GPU barrier is needed.
// A spin that exceeds ~2 s sets an error flag and returns instead of hanging the GPU.
#include "internal.h"
#include <stdlib.h>

namespace ppoaf {

constexpr int kPeerThreads = 1024;
constexpr int kPeerMaxRanks = 8;
constexpr int kPeerMaxVec = 2;            // float4 slots per thread held in registers (1 for a 460 K-parameter policy)
// Spin budget of the cross-GPU barriers in SM clocks (PPOAF_PEER_TIMEOUT_S, default 30 s at ~2 GHz).  The host enqueues a
// stream-level collective before the first exchange of every epoch (ppo.py), so the ranks enter the epoch together; the
// budget only has to cover the skew that builds up inside one epoch.
__device__ long long g_spin_limit = 60000000000LL;
#define kSpinLimit g_spin_limit

#ifdef PPOAF_PEER_TIMING
__device__ long long g_peer_stamps[16];
#define PEER_STAMP(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_peer_stamps[k] = clock64(); } while (0)
#else
#define PEER_STAMP(k) do {} while (0)
#endif

static void configure_spin_limit() {
    static bool done = false;
    if (done) return;
    done = true;
    const char* e = getenv("PPOAF_PEER_TIMEOUT_S");
    if (!e) return;
    const double sec = atof(e);
    if (sec <= 0.0) return;
    const long long clk = (long long)(sec * 2.0e9);
    cudaMemcpyToSymbol(g_spin_limit, &clk, sizeof(clk));
}

struct PeerArgs {
    const float* peer_grads[kPeerMaxRanks];   // the slot holding rank r's gradients for THIS parity (index = rank)
    uint32_t* peer_flags[kPeerMaxRanks];      // flag array of every rank; element [src_rank] is written by src_rank
    uint32_t* local_flags;                    // == peer_flags[my_rank]
    int n_ranks, my_rank;
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

// ctrl (local, zero-initialised): [0] epoch (barrier value of the last call), [2] grid-barrier "go" word, [3] ticket,
// [4] error flag, [8..] beta-power cache (store_beta_powers);
// arrive (local, zero-initialised): one word per CTA (grid barriers of the NVLS variant; the peer kernel counts on ctrl[2])
__global__ void __launch_bounds__(kPeerThreads)
peer_allreduce_adam_kernel(const PeerArgs pa, float* __restrict__ params, float* __restrict__ m, float* __restrict__ v,
                           int64_t n_actor, int64_t n_total, const double* __restrict__ hp,
                           int64_t* __restrict__ adam_step, int32_t* __restrict__ mb_cursor,
                           double* __restrict__ partials, uint32_t* __restrict__ arrive, uint32_t* __restrict__ ctrl) {
    __shared__ double s_scr[32];
    __shared__ double s_pw[2];
    __shared__ float s_f[8];
    __shared__ int s_err;
    const int tid = threadIdx.x;
    const int R = pa.n_ranks;
    double* pw = reinterpret_cast<double*>(ctrl + 8);   // cached (t, beta1, beta2, beta1^t, beta2^t)
    PEER_STAMP(0);
    // ---- 0. before the dependency wait: parameters and moments (only ever written by this kernel) ----
    const int64_t nv = n_total / 4, na = n_actor / 4;
    const int64_t stride = int64_t(gridDim.x) * blockDim.x;
    float4* p4 = reinterpret_cast<float4*>(params);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);
    float4 P[kPeerMaxVec], M[kPeerMaxVec], V[kPeerMaxVec];
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = int64_t(blockIdx.x) * blockDim.x + tid + k * stride;
        if (i < nv) { P[k] = p4[i]; M[k] = m4[i]; V[k] = v4[i]; }
    }
    pdl_wait();                                // the backward pass of this rank has completed: its pushes are out
    pdl_trigger();
    const uint32_t epoch = ctrl[0] + 1;        // every CTA reads the value of the previous call (updated at the very end)
    if (tid == 0) s_err = 0;

    // ---- 1. cross-GPU barrier: publish, then wait for every rank's flag to reach `epoch` ----
    if (blockIdx.x == 0 && tid < R) {
        __threadfence_system();                // this rank's gradient writes (previous kernels) are visible system-wide
        st_release_sys(pa.peer_flags[tid] + pa.my_rank, epoch);
    }
    if (tid < R) {
        const long long t0 = clock64();
        while (int32_t(ld_acquire_sys(pa.local_flags + tid) - epoch) < 0) {
            if (clock64() - t0 > kSpinLimit) { s_err = 1; break; }
        }
    }
    __syncthreads();
    if (s_err) {                               // a peer never arrived: report instead of hanging
        if (tid == 0) atomicExch(ctrl + 4, 1u);
        return;
    }

    PEER_STAMP(1);
    // ---- 2. one-shot reduce in rank order, gradient kept in registers ----
    float4 g[kPeerMaxVec];
    double sa = 0.0, sc = 0.0;
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = int64_t(blockIdx.x) * blockDim.x + tid + k * stride;
        g[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < nv) {
            float4 x[kPeerMaxRanks];               // all R loads (local + NVLink) are issued before any is consumed
#pragma unroll
            for (int r = 0; r < kPeerMaxRanks; ++r)
                if (r < R) x[r] = reinterpret_cast<const float4*>(pa.peer_grads[r])[i];
            float4 acc = x[0];
#pragma unroll
            for (int r = 1; r < kPeerMaxRanks; ++r)
                if (r < R) { acc.x += x[r].x; acc.y += x[r].y; acc.z += x[r].z; acc.w += x[r].w; }
            g[k] = acc;
            const float q = fmaf(acc.x, acc.x, fmaf(acc.y, acc.y, fmaf(acc.z, acc.z, acc.w * acc.w)));
            if (i < na) sa += double(q); else sc += double(q);
        }
    }
    PEER_STAMP(2);
    sa = block_sum(sa, s_scr);
    sc = block_sum(sc, s_scr);
    PEER_STAMP(3);

    // ---- 3. local grid barrier + fixed-order fold of the CTA partials ----
    // flat counter: every CTA adds one with a fire-and-forget red.release and polls the same word until it reads
    // epoch * grid (the grid is the same for every call on these control words, so the count carries over like the epoch).
    // Measured in the one-launch step kernel (DESIGN.md 3.4): 2.5 K clk, against 5.5 K for an arrival word per CTA
    // gathered by CTA 0 plus a release word; an atomicAdd that RETURNS a value costs ~4000 clk at 148 CTAs.
    if (tid == 0) {
        partials[2 * blockIdx.x] = sa;
        partials[2 * blockIdx.x + 1] = sc;
        const uint32_t target = epoch * gridDim.x;
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctrl + 2) : "memory");
        const long long t0 = clock64();
        while (int32_t(ld_acquire_gpu(ctrl + 2) - target) < 0) {
            if (clock64() - t0 > kSpinLimit) { s_err = 1; break; }
        }
    }
    __syncthreads();
    if (s_err) {
        if (tid == 0) atomicExch(ctrl + 4, 2u);
        return;
    }
    PEER_STAMP(4);
    double ta = 0.0, tc = 0.0;
    for (int b = tid; b < int(gridDim.x); b += blockDim.x) { ta += __ldcg(&partials[2 * b]); tc += __ldcg(&partials[2 * b + 1]); }
    ta = block_sum(ta, s_scr);
    tc = block_sum(tc, s_scr);

    PEER_STAMP(5);
    // ---- 4. scalars, then Adam on the register-held gradient ----
    const int64_t t = *adam_step + 1;
    if (tid == 0) {
        const float inv_world = float(hp[PPOAF_HP_INV_WORLD]);
        const float max_norm = float(hp[PPOAF_HP_GRAD_CLIP]);
        const float ca = clip_coef(max_norm, ta, double(inv_world));   // clip_grad_norm_ on the AVERAGED gradient
        const float cc = clip_coef(max_norm, tc, double(inv_world));
        const double b1d = hp[PPOAF_HP_BETA1], b2d = hp[PPOAF_HP_BETA2];
        double p1, p2;
        beta_powers(pw, t, b1d, b2d, p1, p2);
        s_pw[0] = p1; s_pw[1] = p2;
        s_f[0] = float(-(hp[PPOAF_HP_LR] / (1.0 - p1)));
        s_f[1] = float(sqrt(1.0 - p2));
        s_f[2] = float(1.0 - b1d);
        s_f[3] = float(b2d);
        s_f[4] = float(1.0 - b2d);
        s_f[5] = float(hp[PPOAF_HP_ADAM_EPS]);
        s_f[6] = ca;
        s_f[7] = cc;
    }
    __syncthreads();
    PEER_STAMP(6);
    const float neg_step_size = s_f[0], bc2_sqrt = s_f[1], w1 = s_f[2], beta2 = s_f[3], w2 = s_f[4], eps = s_f[5];
    const float inv_world = float(hp[PPOAF_HP_INV_WORLD]);
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = int64_t(blockIdx.x) * blockDim.x + tid + k * stride;
        if (i >= nv) continue;
        const float coef = i < na ? s_f[6] : s_f[7];
        const float4 pq = P[k], mq = M[k], vq = V[k];
        float gg[4] = {g[k].x, g[k].y, g[k].z, g[k].w}, p[4] = {pq.x, pq.y, pq.z, pq.w};
        float mm[4] = {mq.x, mq.y, mq.z, mq.w}, vv[4] = {vq.x, vq.y, vq.z, vq.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {          // same operation order as adam_update_kernel / torch's CPU kernels
            const float gk = __fmul_rn(__fmul_rn(gg[j], inv_world), coef);
            mm[j] = __fadd_rn(mm[j], __fmul_rn(w1, __fsub_rn(gk, mm[j])));
            vv[j] = __fadd_rn(__fmul_rn(vv[j], beta2), __fmul_rn(__fmul_rn(w2, gk), gk));
            float sq;                                  // approximate sqrt / divisions: same arithmetic as optim.cu (adam_vec)
            asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(vv[j]));
            const float denom = __fadd_rn(__fdividef(sq, bc2_sqrt), eps);
            p[j] = __fadd_rn(p[j], __fdividef(__fmul_rn(neg_step_size, mm[j]), denom));
        }
        p4[i] = make_float4(p[0], p[1], p[2], p[3]);
        m4[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
        v4[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
    }
    PEER_STAMP(7);
    // ---- the last CTA to finish advances the counters (everyone has read adam_step / ctrl[0] by then) ----
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(ctrl + 3, 1u) == gridDim.x - 1) {
            *adam_step = t;
            if (mb_cursor) *mb_cursor += 1;
            store_beta_powers(pw, t, hp[PPOAF_HP_BETA1], hp[PPOAF_HP_BETA2], s_pw[0], s_pw[1]);
            ctrl[0] = epoch;
            ctrl[3] = 0u;
        }
    }
}


// =====================================================================================================================
// NVLS variant (NVSwitch multicast): two-shot all-reduce fused with clip + Adam, ZeRO-style ownership.
// The gradient buffers, a parameter staging buffer and a small flag block live in SYMMETRIC memory (same layout on
// every rank, mapped by torch.distributed._symmetric_memory; `*_mc` are multicast addresses of the same buffers).
// Rank r owns slice r of the flat parameter vector:
//   1. cross-GPU barrier (gradients of step t are complete everywhere);
//   2. multimem.ld_reduce over the owned slice: the switch returns the sum over all R replicas, every element is
//      reduced exactly once (by its owner), so all ranks end up with bit-identical parameters by construction;
//   3. slice sums of squares -> exchanged through the flag block (second barrier) -> identical norms everywhere;
//   4. clip + Adam on the owned slice (m, v are only maintained for the owned slice), new parameters go to the owner's
//      staging buffer (a multimem.st broadcast was measured slower: its system fence costs ~10 us);
//   5. third barrier, then every rank gathers all slices from their owners' staging buffers over NVLink.
// Per step and rank this moves ~2 x 4 B/parameter over NVLink regardless of R (the push exchange moves (R-1) x 4 B).
struct NvlsArgs {
    const float* g_mc;                        // multicast address of the gradient buffer of THIS parity
    float* s_local;                           // this rank's parameter staging buffer (holds its own slice)
    const float* s_peer[kPeerMaxRanks];       // staging buffer of rank r (mapped)
    uint32_t* blk_peer[kPeerMaxRanks];        // flag block of rank r (mapped): u32 flags[3][8] | double part[8][2]
    uint32_t* blk_local;
    int n_ranks, my_rank;
};
constexpr int kNvlsPartOff = 128 / 4;         // offset of the partial-sum slots inside a flag block, in u32 words

__device__ __forceinline__ float4 multimem_ld_reduce_f4(const float* mc) {
    float4 r;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
    return r;
}
__device__ __forceinline__ void multimem_st_f4(float* mc, const float4& v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w)
                 : "memory");
}
// every thread tid < R of the calling CTA polls one LOCAL flag word until it reaches `epoch`
__device__ __forceinline__ void xgpu_wait(const uint32_t* flags, int R, uint32_t epoch, int tid, int* s_err) {
    if (tid < R) {
        const long long t0 = clock64();
        while (int32_t(ld_acquire_sys(flags + tid) - epoch) < 0) {
            if (clock64() - t0 > kSpinLimit) { *s_err = 1; break; }
        }
    }
    __syncthreads();
}
// CTA b announces `epoch` in its arrival word; CTA 0 waits for all of them (its threads poll one word each)
// (sys_fence: the CTA's earlier stores must be visible to other GPUs before anything CTA 0 publishes afterwards; one
// cumulative fence by thread 0 after the CTA barrier covers the whole CTA)
__device__ __forceinline__ void gather_to_cta0(uint32_t* arrive, uint32_t epoch, int tid, int* s_err, bool sys_fence = false) {
    __syncthreads();
    if (tid == 0) {
        if (sys_fence) __threadfence_system();
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(arrive + blockIdx.x), "r"(epoch) : "memory");
    }
    if (blockIdx.x == 0) {
        if (tid < int(gridDim.x)) {
            const long long t0 = clock64();
            while (int32_t(ld_acquire_gpu(arrive + tid) - epoch) < 0) {
                if (clock64() - t0 > kSpinLimit) { *s_err = 1; break; }
            }
        }
        __syncthreads();
    }
}

// ctrl (local, zero-initialised): [0] epoch, [3] ticket, [4] error flag, [8..] beta-power cache (store_beta_powers)
// arrive: 2 x gridDim.x local words; partials: 2 doubles per CTA
__global__ void __launch_bounds__(kPeerThreads)
nvls_allreduce_adam_kernel(const NvlsArgs pa, float* __restrict__ params, float* __restrict__ m, float* __restrict__ v,
                           int64_t n_actor, int64_t n_total, const double* __restrict__ hp,
                           int64_t* __restrict__ adam_step, int32_t* __restrict__ mb_cursor,
                           double* __restrict__ partials, uint32_t* __restrict__ arrive, uint32_t* __restrict__ ctrl) {
    __shared__ double s_scr[32];
    __shared__ double s_pw[2];
    __shared__ double s_tot[2];
    __shared__ float s_f[8];
    __shared__ int s_err;
    const int tid = threadIdx.x;
    const int R = pa.n_ranks, me = pa.my_rank;
    double* pw = reinterpret_cast<double*>(ctrl + 8);
    const int64_t nv = n_total / 4, na = n_actor / 4;
    const int64_t slice = (nv + R - 1) / R;
    const int64_t s_lo = int64_t(me) * slice, s_hi = min(nv, s_lo + slice);
    const int64_t gstride = int64_t(gridDim.x) * blockDim.x;
    const int64_t gtid = int64_t(blockIdx.x) * blockDim.x + tid;
    float4* p4 = reinterpret_cast<float4*>(params);
    float4* m4 = reinterpret_cast<float4*>(m);
    float4* v4 = reinterpret_cast<float4*>(v);

    // ---- 0. before the dependency wait: parameters and moments of the owned slice ----
    float4 P[kPeerMaxVec], M[kPeerMaxVec], V[kPeerMaxVec], g[kPeerMaxVec];
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = s_lo + gtid + k * gstride;
        if (i < s_hi) { P[k] = p4[i]; M[k] = m4[i]; V[k] = v4[i]; }
    }
    pdl_wait();
    pdl_trigger();
    PEER_STAMP(0);
    const uint32_t epoch = ctrl[0] + 1;
    if (tid == 0) s_err = 0;
    __syncthreads();

    // ---- 1. cross-GPU barrier: everyone's gradients of this step are complete ----
    if (blockIdx.x == 0 && tid < R) {
        __threadfence_system();
        st_release_sys(pa.blk_peer[tid] + 0 * 8 + me, epoch);
    }
    xgpu_wait(pa.blk_local + 0 * 8, R, epoch, tid, &s_err);
    if (s_err) { if (tid == 0) atomicExch(ctrl + 4, 1u); return; }

    PEER_STAMP(1);
    // ---- 2. in-switch reduction of the owned slice ----
    double sa = 0.0, sc = 0.0;
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = s_lo + gtid + k * gstride;
        g[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (i < s_hi) {
            g[k] = multimem_ld_reduce_f4(pa.g_mc + 4 * i);
            const float q = fmaf(g[k].x, g[k].x, fmaf(g[k].y, g[k].y, fmaf(g[k].z, g[k].z, g[k].w * g[k].w)));
            if (i < na) sa += double(q); else sc += double(q);
        }
    }
    PEER_STAMP(2);
    sa = block_sum(sa, s_scr);
    sc = block_sum(sc, s_scr);
    if (tid == 0) { partials[2 * blockIdx.x] = sa; partials[2 * blockIdx.x + 1] = sc; }

    // ---- 3. slice sums -> every rank (CTA 0 folds the CTA partials and writes them into every peer's flag block) ----
    gather_to_cta0(arrive, epoch, tid, &s_err);
    if (blockIdx.x == 0) {
        double ta = 0.0, tc = 0.0;
        for (int b = tid; b < int(gridDim.x); b += blockDim.x) { ta += __ldcg(&partials[2 * b]); tc += __ldcg(&partials[2 * b + 1]); }
        ta = block_sum(ta, s_scr);
        tc = block_sum(tc, s_scr);
        if (tid < R) {
            double* slot = reinterpret_cast<double*>(pa.blk_peer[tid] + kNvlsPartOff) + 2 * me;
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(slot), "d"(ta) : "memory");
            asm volatile("st.relaxed.sys.global.f64 [%0], %1;" ::"l"(slot + 1), "d"(tc) : "memory");
            st_release_sys(pa.blk_peer[tid] + 1 * 8 + me, epoch);
        }
    }
    xgpu_wait(pa.blk_local + 1 * 8, R, epoch, tid, &s_err);
    if (s_err) { if (tid == 0) atomicExch(ctrl + 4, 2u); return; }
    if (tid == 0) {
        const double* part = reinterpret_cast<const double*>(pa.blk_local + kNvlsPartOff);
        double ta = 0.0, tc = 0.0;
        for (int r = 0; r < R; ++r) {                  // rank order: identical everywhere
            double xa, xc;
            asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(xa) : "l"(part + 2 * r) : "memory");
            asm volatile("ld.relaxed.sys.global.f64 %0, [%1];" : "=d"(xc) : "l"(part + 2 * r + 1) : "memory");
            ta += xa; tc += xc;
        }
        s_tot[0] = ta; s_tot[1] = tc;
    }
    __syncthreads();

    PEER_STAMP(3);
    // ---- 4. scalars, Adam on the owned slice, broadcast of the new parameters ----
    const int64_t t = *adam_step + 1;
    const float inv_world = float(hp[PPOAF_HP_INV_WORLD]);
    if (tid == 0) {
        const float max_norm = float(hp[PPOAF_HP_GRAD_CLIP]);
        const float ca = clip_coef(max_norm, s_tot[0], double(inv_world));
        const float cc = clip_coef(max_norm, s_tot[1], double(inv_world));
        const double b1d = hp[PPOAF_HP_BETA1], b2d = hp[PPOAF_HP_BETA2];
        double p1, p2;
        beta_powers(pw, t, b1d, b2d, p1, p2);
        s_pw[0] = p1; s_pw[1] = p2;
        s_f[0] = float(-(hp[PPOAF_HP_LR] / (1.0 - p1)));
        s_f[1] = float(sqrt(1.0 - p2));
        s_f[2] = float(1.0 - b1d);
        s_f[3] = float(b2d);
        s_f[4] = float(1.0 - b2d);
        s_f[5] = float(hp[PPOAF_HP_ADAM_EPS]);
        s_f[6] = ca;
        s_f[7] = cc;
    }
    __syncthreads();
    const float neg_step_size = s_f[0], bc2_sqrt = s_f[1], w1 = s_f[2], beta2 = s_f[3], w2 = s_f[4], eps = s_f[5];
#pragma unroll
    for (int k = 0; k < kPeerMaxVec; ++k) {
        const int64_t i = s_lo + gtid + k * gstride;
        if (i >= s_hi) continue;
        const float coef = i < na ? s_f[6] : s_f[7];
        float gg[4] = {g[k].x, g[k].y, g[k].z, g[k].w}, p[4] = {P[k].x, P[k].y, P[k].z, P[k].w};
        float mm[4] = {M[k].x, M[k].y, M[k].z, M[k].w}, vv[4] = {V[k].x, V[k].y, V[k].z, V[k].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {          // same operation order as adam_update_kernel / torch's CPU kernels
            const float gk = __fmul_rn(__fmul_rn(gg[j], inv_world), coef);
            mm[j] = __fadd_rn(mm[j], __fmul_rn(w1, __fsub_rn(gk, mm[j])));
            vv[j] = __fadd_rn(__fmul_rn(vv[j], beta2), __fmul_rn(__fmul_rn(w2, gk), gk));
            float sq;                                  // approximate sqrt / divisions: same arithmetic as optim.cu (adam_vec)
            asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(vv[j]));
            const float denom = __fadd_rn(__fdividef(sq, bc2_sqrt), eps);
            p[j] = __fadd_rn(p[j], __fdividef(__fmul_rn(neg_step_size, mm[j]), denom));
        }
        m4[i] = make_float4(mm[0], mm[1], mm[2], mm[3]);
        v4[i] = make_float4(vv[0], vv[1], vv[2], vv[3]);
        reinterpret_cast<float4*>(pa.s_local)[i] = make_float4(p[0], p[1], p[2], p[3]);
    }

    PEER_STAMP(4);
    // ---- 5. third barrier: every rank's slice has landed in every staging buffer ----
    // the staging stores become visible GPU-wide through the release below; the peers read them from this GPU's L2, so
    // the only system-scope ordering needed is CTA 0's cumulative release of the flag (a per-CTA fence.sys cost ~10 us)
    gather_to_cta0(arrive + gridDim.x, epoch, tid, &s_err);
    if (blockIdx.x == 0 && tid < R) {
        __threadfence_system();
        st_release_sys(pa.blk_peer[tid] + 2 * 8 + me, epoch);
    }
    xgpu_wait(pa.blk_local + 2 * 8, R, epoch, tid, &s_err);
    if (s_err) { if (tid == 0) atomicExch(ctrl + 4, 3u); return; }
    PEER_STAMP(5);
    for (int64_t i = gtid; i < nv; i += gstride) {           // every slice straight from its owner's staging buffer
        const int owner = int(i / slice);
        float4 x;
        asm volatile("ld.relaxed.sys.global.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w) : "l"(reinterpret_cast<const float4*>(pa.s_peer[owner]) + i) : "memory");
        p4[i] = x;
    }
    PEER_STAMP(6);

    // ---- the last CTA to finish advances the counters ----
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        if (atomicAdd(ctrl + 3, 1u) == gridDim.x - 1) {
            *adam_step = t;
            if (mb_cursor) *mb_cursor += 1;
            store_beta_powers(pw, t, hp[PPOAF_HP_BETA1], hp[PPOAF_HP_BETA2], s_pw[0], s_pw[1]);
            ctrl[0] = epoch;
            ctrl[3] = 0u;
        }
    }
}

}  // namespace ppoaf

using namespace ppoaf;

// ---- peer-memory plumbing (cudaMalloc + CUDA IPC; the handles travel through torch.distributed) ----------
extern "C" int ppoaf_peer_alloc(size_t bytes, void** out) {
    configure_spin_limit();            // set-up call: never inside a stream capture
    PPOAF_CHECK_ARG(out != nullptr && bytes > 0, "ppoaf_peer_alloc: bad arguments");
    cudaError_t e = cudaMalloc(out, bytes);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_alloc: cudaMalloc failed: %s", cudaGetErrorString(e));
    e = cudaMemset(*out, 0, bytes);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_alloc: cudaMemset failed: %s", cudaGetErrorString(e));
    return 0;
}
extern "C" int ppoaf_peer_free(void* p) {
    cudaError_t e = cudaFree(p);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_free: %s", cudaGetErrorString(e));
    return 0;
}
extern "C" int ppoaf_peer_export(void* p, uint8_t* handle64) {
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    cudaError_t e = cudaIpcGetMemHandle(&h, p);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_export: cudaIpcGetMemHandle failed: %s", cudaGetErrorString(e));
    memcpy(handle64, &h, 64);
    return 0;
}
extern "C" int ppoaf_peer_import(const uint8_t* handle64, void** out) {
    cudaIpcMemHandle_t h;
    memcpy(&h, handle64, 64);
    cudaError_t e = cudaIpcOpenMemHandle(out, h, cudaIpcMemLazyEnablePeerAccess);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_import: cudaIpcOpenMemHandle failed: %s", cudaGetErrorString(e));
    return 0;
}
extern "C" int ppoaf_peer_close(void* p) {
    cudaError_t e = cudaIpcCloseMemHandle(p);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_peer_close: %s", cudaGetErrorString(e));
    return 0;
}

static size_t peer_arrive_bytes() { return align_up(size_t(sm_count()) * sizeof(uint32_t), 256); }
constexpr size_t kCtrlWordsBytes = 256;    // the control words of both kernels: 8 u32 words, then the beta-power cache
static_assert(8 * sizeof(uint32_t) + kBetaCacheDoubles * sizeof(double) <= kCtrlWordsBytes,
              "the beta-power cache must fit the control words");
extern "C" size_t ppoaf_peer_ctrl_bytes(void) {
    return size_t(sm_count()) * 2 * sizeof(double) + peer_arrive_bytes() + kCtrlWordsBytes;
}

// peer_grads[r] / peer_flags[r]: pointers valid on THIS device for rank r's buffers (own rank: the local pointers).
// ctrl: local zero-initialised scratch of ppoaf_peer_ctrl_bytes() bytes (CTA partials | arrival words | control words).
extern "C" int ppoaf_peer_allreduce_adam(const void* const* peer_grads, void* const* peer_flags, int32_t n_ranks,
                                         int32_t my_rank, float* params, float* adam_m, float* adam_v,
                                         int64_t* adam_step, int32_t* mb_cursor, const double* hparams,
                                         int64_t n_actor, int64_t n_critic, void* ctrl, void* stream) {
    PPOAF_CHECK_ARG(n_ranks >= 1 && n_ranks <= kPeerMaxRanks && my_rank >= 0 && my_rank < n_ranks,
                    "ppoaf_peer_allreduce_adam: up to %d ranks", kPeerMaxRanks);
    PPOAF_CHECK_ARG(n_actor % 4 == 0 && n_critic % 4 == 0, "ppoaf_peer_allreduce_adam: segments must be multiples of 4 floats");
    const int64_t n_total = n_actor + n_critic;
    int grid = sm_count();
    const int64_t need = ceil_div64(n_total / 4, kPeerThreads);
    if (need < grid) grid = int(need < 1 ? 1 : need);
    PPOAF_CHECK_ARG(n_total / 4 <= int64_t(grid) * kPeerThreads * kPeerMaxVec,
                    "ppoaf_peer_allreduce_adam: %lld parameters exceed the register-resident limit; use the NCCL path",
                    (long long)n_total);
    PeerArgs pa{};
    for (int r = 0; r < n_ranks; ++r) {
        pa.peer_grads[r] = static_cast<const float*>(peer_grads[r]);
        pa.peer_flags[r] = static_cast<uint32_t*>(peer_flags[r]);
    }
    pa.local_flags = static_cast<uint32_t*>(peer_flags[my_rank]);
    pa.n_ranks = n_ranks;
    pa.my_rank = my_rank;
    double* partials = static_cast<double*>(ctrl);
    uint32_t* arrive = reinterpret_cast<uint32_t*>(static_cast<char*>(ctrl) + size_t(sm_count()) * 2 * sizeof(double));
    uint32_t* words = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(arrive) + peer_arrive_bytes());
    // chained like the single-rank optimizer: the launch before it (last backward GEMM) never writes params / m / v
    launch_chain(peer_allreduce_adam_kernel, dim3(grid), dim3(kPeerThreads), 0, (cudaStream_t)stream, pa, params, adam_m,
                 adam_v, n_actor, n_total, hparams, adam_step, mb_cursor, partials, arrive, words);
    PPOAF_CHECK_LAUNCH("peer_allreduce_adam_kernel");
    return 0;
}

#ifdef PPOAF_PEER_TIMING
extern "C" int ppoaf_debug_peer_stamps(long long* out_host) {
    return cudaMemcpyFromSymbol(out_host, ppoaf::g_peer_stamps, sizeof(long long) * 16) == cudaSuccess ? 0 : 1;
}
#endif

// ---- NVLS variant ------------------------------------------------------------------------------------------------
extern "C" size_t ppoaf_nvls_ctrl_bytes(void) { configure_spin_limit();
    return size_t(sm_count()) * 2 * sizeof(double) + 2 * peer_arrive_bytes() + kCtrlWordsBytes;
}
extern "C" size_t ppoaf_nvls_flag_block_bytes(void) { return 256; }

// g_mc: multicast address of this parity's gradient buffer; staging[r]: rank r's parameter staging buffer mapped on
// this device; flag_blocks[r]: rank r's zero-initialised flag block mapped on this device
// (ppoaf_nvls_flag_block_bytes() bytes, symmetric memory); ctrl: local zeroed scratch of ppoaf_nvls_ctrl_bytes().
extern "C" int ppoaf_nvls_allreduce_adam(const float* g_mc, void* const* staging, void* const* flag_blocks,
                                         int32_t n_ranks, int32_t my_rank, float* params, float* adam_m, float* adam_v,
                                         int64_t* adam_step, int32_t* mb_cursor, const double* hparams, int64_t n_actor,
                                         int64_t n_critic, void* ctrl, void* stream) {
    PPOAF_CHECK_ARG(n_ranks >= 2 && n_ranks <= kPeerMaxRanks && my_rank >= 0 && my_rank < n_ranks,
                    "ppoaf_nvls_allreduce_adam: 2..%d ranks", kPeerMaxRanks);
    PPOAF_CHECK_ARG(n_actor % 4 == 0 && n_critic % 4 == 0, "ppoaf_nvls_allreduce_adam: segments must be multiples of 4 floats");
    PPOAF_CHECK_ARG(g_mc && staging && flag_blocks, "ppoaf_nvls_allreduce_adam: null pointers");
    const int64_t n_total = n_actor + n_critic;
    const int64_t nv = n_total / 4;
    const int64_t slice = (nv + n_ranks - 1) / n_ranks;
    int grid = sm_count();
    const int64_t need = ceil_div64(slice, kPeerThreads);
    if (need < grid) grid = int(need < 1 ? 1 : need);
    PPOAF_CHECK_ARG(slice <= int64_t(grid) * kPeerThreads * kPeerMaxVec,
                    "ppoaf_nvls_allreduce_adam: %lld parameters exceed the register-resident limit", (long long)n_total);
    NvlsArgs pa{};
    pa.g_mc = g_mc;
    pa.s_local = static_cast<float*>(staging[my_rank]);
    for (int r = 0; r < n_ranks; ++r) {
        pa.blk_peer[r] = static_cast<uint32_t*>(flag_blocks[r]);
        pa.s_peer[r] = static_cast<const float*>(staging[r]);
    }
    pa.blk_local = static_cast<uint32_t*>(flag_blocks[my_rank]);
    pa.n_ranks = n_ranks; pa.my_rank = my_rank;
    double* partials = static_cast<double*>(ctrl);
    uint32_t* arrive = reinterpret_cast<uint32_t*>(static_cast<char*>(ctrl) + size_t(sm_count()) * 2 * sizeof(double));
    uint32_t* words = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(arrive) + 2 * peer_arrive_bytes());
    // arrive is used as two arrays of gridDim.x words: the second one starts at arrive + grid
    launch_chain(nvls_allreduce_adam_kernel, dim3(grid), dim3(kPeerThreads), 0, (cudaStream_t)stream, pa, params, adam_m,
                 adam_v, n_actor, n_total, hparams, adam_step, mb_cursor, partials, arrive, words);
    PPOAF_CHECK_LAUNCH("nvls_allreduce_adam_kernel");
    return 0;
}

