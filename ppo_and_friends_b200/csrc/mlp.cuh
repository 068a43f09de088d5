// fp32 grouped-GEMM core for the actor/critic MLP layers at reference minibatch sizes (B = 128..512,
// hidden 64..512).  One layer of one network is ~30-50 MFLOP: far too small to be a dense
// tensor-core contraction (SURVEY.md §8d), and a minibatch step is a chain of ~10 dependent phases,
// so the design goal is latency per phase and launches per step, not peak FLOP/s:
//
//   * GROUPED launches: one launch computes every GEMM of a phase (actor and critic forward layer l;
//     or dW and dX of layer l for both networks), so a step is 8 GEMM launches instead of 22 and
//     each launch fills the 148 SMs with 32x64 output tiles;
//   * 256 threads per CTA = 8 warps; each warp owns a CONTIGUOUS 1/8 slice of the reduction dimension
//     and computes the whole 32x64 tile over it with an 8x8 register microtile (intra-CTA split-K;
//     the 8 partial tiles are summed through shared memory).  16 LDS.128 feed 256 FFMA;
//   * every warp runs its OWN cp.async ring (4 slots of 8 k's, all of them issued before the first
//     FFMA) and synchronises only with __syncwarp: there is no CTA-wide barrier in the main loop, so
//     the warps of an SM drift apart and one warp's shared-memory loads hide behind the others' FFMAs;
//   * 96 KB of shared memory and <= 128 registers per thread: two CTAs share an SM, so a launch of up
//     to 296 tiles is ONE wave (the backward launches have 192);
//   * operands stay in their GLOBAL orientation (so 16-byte cp.async serves all three GEMM flavours,
//     with zero-fill for ragged edges);
//   * fused epilogues (bias + activation; activation derivative; bias gradient + per-tile sum of
//     squares for the gradient-norm clip) and a fused row gather on the operand indexed by sample,
//     so the gathered minibatch never exists in HBM.
//
//   forward      Y[m,n]  = act(sum_k X[idx[m],k] W[n,k] + b[n])        FeedForwardNetwork.forward
//   backward-x   dX[m,k] = (sum_n dZ[m,n] W[n,k]) * act'(Xact[m,k])    autograd of the same
//   backward-w   dW[n,k] = sum_m dZ[m,n] X[idx[m],k] ; db[n] = sum_m dZ[m,n]
#pragma once
#include "common.cuh"

namespace ppoaf {

__device__ __forceinline__ float act_fwd(float x, int act) {
    switch (act) {
        case PPOAF_ACT_RELU: return x > 0.f ? x : 0.f;
        case PPOAF_ACT_LEAKY_RELU: return x > 0.f ? x : 0.01f * x;
        case PPOAF_ACT_TANH: return tanhf(x);
        case PPOAF_ACT_IDENTITY: return x;
        default: return act_fwd_ext(x, act);
    }
}
// derivative expressed through the activation OUTPUT y (sign(y) == sign(x) for relu / leaky relu); ids 8-11 (stored
// derivative) pass act'(z) itself as y
__device__ __forceinline__ float act_bwd_from_out(float y, int act) {
    switch (act) {
        case PPOAF_ACT_RELU: return y > 0.f ? 1.f : 0.f;
        case PPOAF_ACT_LEAKY_RELU: return y > 0.f ? 1.f : 0.01f;
        case PPOAF_ACT_TANH: return 1.f - y * y;
        case PPOAF_ACT_IDENTITY: return 1.f;
        default: return act_bwd_ext(y, act);
    }
}

// EPI_FWD_DACT: EPI_FWD that also stores act'(z) to GemmProblem::dact (act_stores_derivative ids, FFMA tiles only)
enum { EPI_FWD = 0, EPI_BWD_X = 1, EPI_BWD_W = 2, EPI_FWD_DACT = 3 };
constexpr int kMaxGroup = 6;

struct GemmProblem {
    const float* A; const float* B; float* C;
    const float* bias;              // EPI_FWD: bias[n]
    const float* aux;               // EPI_BWD_X: activation output of the layer below, aux[m*ldaux + n] (its stored
                                    //   act'(z) for act_stores_derivative ids)
    union {                         // (one slot: the struct, and the launches' parameter blocks, keep their size)
        float* dact;                // EPI_FWD_DACT: act'(z) out, dact[m*ldc + n]
        float* dbias;               // EPI_BWD_W: dbias[m] = sum_r A(m, r)
    };
    double* sq_out;                 // EPI_BWD_W: sq_out[tile] = sum of squares of this tile of dW (+ db), or null
    const int64_t* idxA;            // optional row indirection on A's row index
    const int64_t* idxB;            // optional row indirection on B's row index
    int lda, ldb, ldc, ldaux;       // A(m,r): A_RC ? A[row(m)*lda + r] : A[row(r)*lda + m];  B likewise with n
    int M, N, K;                    // C is M x N, reduction length K
    int act;
    int flavour;                    // epi * 4 + (VA == 4) * 2 + (VB == 4)
    int tiles_n;                    // number of tiles along N
    int tile_begin;                 // first linear tile id of this problem inside the launch
    int b_static;                   // B is not written by the launch right before this one (and has no gather): it may
                                    //   be staged before the programmatic-dependency wait
    int bn;                         // fused_step.cu: tile width along N chosen for this problem's phase (16 / 32)
    int a_par, b_par;               // fused_step.cu: operand rows to skip on odd steps (double-buffered gathered minibatch rows)
};
struct MirrorSet {                   // peer copies of the gradient buffer (R > 1 push exchange): byte offsets from
    int n;                           //   a local gradient address to the same element in every peer's receive slot
    long long delta[PPOAF_MAX_MIRROR];
};
template <typename T>
__device__ __forceinline__ void mirror_store(const MirrorSet& mir, T* local, const T& v) {
    for (int q = 0; q < mir.n; ++q) *reinterpret_cast<T*>(reinterpret_cast<char*>(local) + mir.delta[q]) = v;
}
struct GroupedGemmArgs {
    int n_problems;
    int cursor_stride;              // idx tables start at (*cursor) * cursor_stride (the minibatch cursor, so
    const int32_t* cursor;          //   one captured graph serves every minibatch); cursor may be null
    GemmProblem p[kMaxGroup];
    MirrorSet mirror;               // applied to the outputs of EPI_BWD_W problems (dW, db)
};

constexpr int kBM = 32, kBN = 64, kThreads = 512, kGroups = 16;
constexpr int kLoadGroups = 4;                  // column groups of a panel: group c = the K slices of warps 4c .. 4c+3
constexpr int kKRound = 512;                    // reduction extent staged per round (a whole panel)
constexpr int kPanelFloats = (kBM + kBN) * (kKRound + 8);     // 49920 floats = 195 KB
constexpr int kRedLd = kBN + 8;                 // 72 = 8 (mod 32): the (ty, tx) lanes of a warp hit 32 distinct banks
constexpr int kRedFloats = kGroups * kBM * kRedLd + kGroups * kBM;
static_assert(kRedFloats <= kPanelFloats, "the split-K reduction reuses the panel memory");
constexpr size_t kGemmSmemBytes = sizeof(float) * size_t(kPanelFloats);

__device__ __forceinline__ unsigned smem_addr(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
__device__ __forceinline__ void cp_async_16(float* smem_dst, const float* gmem_src, bool valid) {
    const int bytes = valid ? 16 : 0;   // src-size 0: the 16 destination bytes are zero-filled
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr(smem_dst)), "l"(gmem_src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cp_async_4(float* smem_dst, const float* gmem_src, bool valid) {
    const int bytes = valid ? 4 : 0;
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(smem_addr(smem_dst)), "l"(gmem_src), "r"(bytes) : "memory");
}
// the mbarrier receives one arrival from this thread once all of its earlier cp.async's have landed
__device__ __forceinline__ void cp_async_arrive(uint64_t* bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(smem_addr(bar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "MBAR_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra MBAR_DONE_%=;\n"
        "bra MBAR_WAIT_%=;\n"
        "MBAR_DONE_%=:\n"
        "}\n" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}

// Panel layout of one operand for one round of Kr reduction indices (Kr4 = Kr rounded up to 4):
//   RC (reduction-contiguous in global, element P[row(out)*ld + k]): panel[out][lds], lds = Kr4 + 4 or 8 so that
//      lds / 4 is odd (rows of a fragment land on distinct 16-byte bank groups)
//   OC (output-contiguous in global,    element P[row(k)*ld + out]): panel[k][OUT]
// Both are staged by ALL threads with lanes running along the contiguous global direction, so every cp.async
// instruction reads whole 128-byte lines and writes them to contiguous shared memory (scattered 16-byte
// destinations cost ~3x: measured, scratch/load_probe.cu).
__device__ __forceinline__ int rc_stride(int Kr4) { return Kr4 + ((Kr4 & 7) == 0 ? 4 : 8); }

__device__ __forceinline__ void cp_async_16_plain(unsigned smem_dst, const float* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}

// Stage columns [k_lo, k_hi) (multiples of 4, relative to the round start k_base) of an RC operand.
// 16 lanes run along k (one 16-byte chunk each), thread rows are fixed: row = tid / 16 (+ 32 for the second half of
// a 64-row operand), so the row pointers (and gather indices) are resolved once per tile.  Rows beyond the operand's
// extent are simply not staged: they only feed outputs that are never stored.
template <int OUT, int V>
struct RcStager {
    const float* rowp[OUT / 32];       // row base + this lane's column offset
    bool ok[OUT / 32];
    __device__ __forceinline__ void plan(const float* __restrict__ P, int ld, const int64_t* __restrict__ idx, int out0,
                                         int out_ext, int tid) {
#pragma unroll
        for (int j = 0; j < OUT / 32; ++j) {
            const int go = out0 + (tid >> 4) + 32 * j;
            ok[j] = go < out_ext;
            const int64_t r = ok[j] ? (idx ? idx[go] : int64_t(go)) : 0;
            rowp[j] = P + r * ld + (tid & 15) * 4;
        }
    }
    __device__ __forceinline__ void stage(float* panel, int lds, int k_base, int K, int k_lo, int k_hi, int tid) const {
        const unsigned dst0 = smem_addr(panel + (tid >> 4) * lds + (tid & 15) * 4);
        for (int kk = k_lo; kk + (tid & 15) * 4 < k_hi; kk += 64) {
#pragma unroll
            for (int j = 0; j < OUT / 32; ++j) {
                if constexpr (V == 4) {                                           // K % 4 == 0: no ragged chunk
                    if (ok[j]) cp_async_16_plain(dst0 + unsigned(32 * j * lds + kk) * 4u, rowp[j] + k_base + kk);
                } else {
                    float* dst = panel + ((tid >> 4) + 32 * j) * lds + (tid & 15) * 4 + kk;
                    const int k = k_base + kk + (tid & 15) * 4;
#pragma unroll
                    for (int e = 0; e < 4; ++e) cp_async_4(dst + e, rowp[j] + k_base + kk + e, ok[j] && k + e < K);
                }
            }
        }
    }
};

// Stage k-rows [k_lo, k_hi) of an OC operand: OUT / 4 lanes run along the contiguous outputs of one k-row.
// k-rows in [K, k_hi) are zero-filled (they are multiplied into valid outputs); columns beyond the operand's extent
// are not staged.  sidx: gather indices of this round's k's staged in shared memory, or null.
template <int OUT, int V>
__device__ __forceinline__ void stage_oc(float* panel, const float* __restrict__ P, int ld, const int* sidx, int out0,
                                         int out_ext, int k_base, int K, int k_lo, int k_hi, int tid) {
    constexpr int CPR = OUT / 4;
    const int o = (tid % CPR) * 4;
    if (V == 4 && out0 + o >= out_ext) return;                                // out_ext % 4 == 0
    const float* base = P + out0 + o;
    float* dst = panel + (k_lo + tid / CPR) * OUT + o;
    for (int kk = k_lo + tid / CPR; kk < k_hi; kk += kThreads / CPR, dst += (kThreads / CPR) * OUT) {
        const bool kok = k_base + kk < K;
        const int64_t r = kok ? (sidx ? int64_t(sidx[kk]) : int64_t(k_base + kk)) : 0;
        const float* src = base + r * ld;
        if constexpr (V == 4) {
            cp_async_16(dst, src, kok);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) cp_async_4(dst + e, src + e, kok && out0 + o + e < out_ext);
        }
    }
}

__device__ __forceinline__ float act_fwd_fast(float x, int act) {
    switch (act) {
        case PPOAF_ACT_RELU: return x > 0.f ? x : 0.f;
        case PPOAF_ACT_LEAKY_RELU: return x > 0.f ? x : 0.01f * x;
        case PPOAF_ACT_TANH: return fast_tanh(x);
        case PPOAF_ACT_IDENTITY: return x;
        default: return act_fwd_ext(x, act);
    }
}

// Position of microtile element i (0..7) of lane-coordinate t inside an operand tile of OUT rows:
//   RC: t + (OUT/8) * i             (consecutive lanes -> consecutive rows: conflict-free LDS.128 along k)
//   OC: two runs of 4 contiguous    (consecutive lanes -> one contiguous 16-byte-per-lane span)
template <int OUT, bool RC>
__device__ __forceinline__ int frag_pos(int t, int i) {
    if constexpr (RC) return t + (OUT / 8) * i;
    else return (i < 4) ? 4 * t + i : OUT / 2 + 4 * t + (i - 4);
}

// f[i][q] = operand(out_i, k + q), 8 outputs x 4 k's.  RC: base = panel + k, stride = lds; OC: base = panel + k * OUT
template <int OUT, bool RC>
__device__ __forceinline__ void load_frag(float (&f)[8][4], const float* base, int lds, int t) {
    if constexpr (RC) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const float4 v = *reinterpret_cast<const float4*>(base + (t + (OUT / 8) * i) * lds);
            f[i][0] = v.x; f[i][1] = v.y; f[i][2] = v.z; f[i][3] = v.w;
        }
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const float4 lo = *reinterpret_cast<const float4*>(base + q * OUT + 4 * t);
            const float4 hi = *reinterpret_cast<const float4*>(base + q * OUT + OUT / 2 + 4 * t);
            f[0][q] = lo.x; f[1][q] = lo.y; f[2][q] = lo.z; f[3][q] = lo.w;
            f[4][q] = hi.x; f[5][q] = hi.y; f[6][q] = hi.z; f[7][q] = hi.w;
        }
    }
}

#ifdef PPOAF_GEMM_TIMING
__device__ long long g_gemm_stamps[16];
#define PPOAF_STAMP(k) do { if (blockIdx.x == 0 && threadIdx.x == 0) g_gemm_stamps[k] = clock64(); } while (0)
#else
#define PPOAF_STAMP(k) do {} while (0)
#endif

__device__ __forceinline__ float4 load4_guarded(const float* p, int remaining, bool vec) {
    if (vec && remaining >= 4) return *reinterpret_cast<const float4*>(p);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (remaining > 0) v.x = p[0];
    if (remaining > 1) v.y = p[1];
    if (remaining > 2) v.z = p[2];
    if (remaining > 3) v.w = p[3];
    return v;
}

// EXT: the epilogues also take activation ids 4-11 (grouped_gemm_ext_kernel)
template <bool A_RC, bool B_RC, int VA, int VB, int EPI, bool EXT>
__device__ __forceinline__ void gemm_tile(const GemmProblem& g, int tile, const int32_t* cursor, int cursor_stride,
                                          const MirrorSet& mir, float* smem, uint64_t* bars, int* s_idx) {
    const int tid = threadIdx.x;
    PPOAF_STAMP(1);
    const int grp = tid >> 5, lane = tid & 31;
    const int tx = lane & 7, ty = lane >> 3;                  // 8 column-lanes x 4 row-lanes per warp
    const int m0 = (tile / g.tiles_n) * kBM, n0 = (tile % g.tiles_n) * kBN;

    // ---- before the dependency wait: a B operand that the previous launch does not write (weights in the forward
    // and backward-x launches, stored activations in backward-w) starts travelling while that launch drains ----
    RcStager<kBN, VB> rcb;
    const bool b_early = g.b_static && !g.idxB;
    if (b_early) {
        const int Kr = min(g.K, kKRound), Kr4 = (Kr + 3) & ~3;
        const int ldsA0 = A_RC ? rc_stride(Kr4) : kBM, ldsB0 = B_RC ? rc_stride(Kr4) : kBN;
        float* panelB0 = smem + (A_RC ? kBM * ldsA0 : Kr4 * kBM);
        if constexpr (B_RC) { rcb.plan(g.B, g.ldb, nullptr, n0, g.N, tid); rcb.stage(panelB0, ldsB0, 0, g.K, 0, Kr4, tid); }
        else stage_oc<kBN, VB>(panelB0, g.B, g.ldb, nullptr, n0, g.N, 0, g.K, 0, Kr4, tid);
    }
    pdl_wait();                                    // everything below may read what the previous launch wrote
    pdl_trigger();                                 // after the wait: the next launch's early reads then only ever
                                                   //   overlap THIS launch, never the one before it
    // the minibatch cursor is only needed by the gathering layers: no dependent global load on the others
    const int64_t idx_off = (cursor && (g.idxA || g.idxB)) ? int64_t(*cursor) * cursor_stride : 0;
    const int64_t* idxA = g.idxA ? g.idxA + idx_off : nullptr;
    const int64_t* idxB = g.idxB ? g.idxB + idx_off : nullptr;

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    float bsum[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) bsum[i] = 0.f;

    // RC operands: row pointers (through the gather indices) once per tile; OC operands: the gather indices of
    // a round's k's are staged in shared memory
    int* s_idx_a = s_idx;                      // [kKRound]
    int* s_idx_b = s_idx + kKRound;            // [kKRound]
    RcStager<kBM, VA> rca;
    if constexpr (A_RC) rca.plan(g.A, g.lda, idxA, m0, g.M, tid);
    if constexpr (B_RC) { if (!b_early) rcb.plan(g.B, g.ldb, idxB, n0, g.N, tid); }

    const int n_rounds = (g.K + kKRound - 1) / kKRound;
#pragma unroll 1
    for (int round = 0; round < n_rounds; ++round) {
        const int k_base = round * kKRound;
        const int Kr = min(g.K - k_base, kKRound);
        const int Kr4 = (Kr + 3) & ~3;
        const int Kw = (((Kr + kGroups - 1) / kGroups) + 3) & ~3;        // k's per warp this round (multiple of 4)
        const int ldsA = A_RC ? rc_stride(Kr4) : kBM, ldsB = B_RC ? rc_stride(Kr4) : kBN;
        float* panelA = smem;
        float* panelB = smem + (A_RC ? kBM * ldsA : Kr4 * kBM);
        if (round > 0) __syncthreads();                    // everyone is done reading the previous round's panel
        if (!A_RC && idxA) for (int k = tid; k < Kr; k += kThreads) s_idx_a[k] = int(idxA[k_base + k]);
        if (!B_RC && idxB) for (int k = tid; k < Kr; k += kThreads) s_idx_b[k] = int(idxB[k_base + k]);
        if ((!A_RC && idxA) || (!B_RC && idxB)) __syncthreads();

        // ---- stage the whole round, column group by column group; completion is signalled asynchronously ----
#pragma unroll 1
        for (int c = 0; c < kLoadGroups; ++c) {
            const int k_lo = min(Kr4, c * (kGroups / kLoadGroups) * Kw);
            const int k_hi = min(Kr4, (c + 1) * (kGroups / kLoadGroups) * Kw);
            if constexpr (A_RC) rca.stage(panelA, ldsA, k_base, g.K, k_lo, k_hi, tid);
            else stage_oc<kBM, VA>(panelA, g.A, g.lda, idxA ? s_idx_a : nullptr, m0, g.M, k_base, g.K, k_lo, k_hi, tid);
            if (!(b_early && round == 0)) {
                if constexpr (B_RC) rcb.stage(panelB, ldsB, k_base, g.K, k_lo, k_hi, tid);
                else stage_oc<kBN, VB>(panelB, g.B, g.ldb, idxB ? s_idx_b : nullptr, n0, g.N, k_base, g.K, k_lo, k_hi, tid);
            }
            cp_async_arrive(&bars[c]);
        }
        if (round == 0) PPOAF_STAMP(2);

        // ---- this warp's K slice: wait for its column group only ----
        const int kbeg = grp * Kw, kend = min(Kr4, kbeg + Kw);
        mbar_wait(&bars[grp / (kGroups / kLoadGroups)], unsigned(round & 1));
        if (round == 0) PPOAF_STAMP(3);
#pragma unroll 1   // one 8x8x4 block (16 LDS.128 + 256 FFMA) is the whole hot loop body
        for (int k = kbeg; k < kend; k += 4) {
            float a[8][4], bf[8][4];
            load_frag<kBM, A_RC>(a, A_RC ? panelA + k : panelA + k * kBM, ldsA, ty);
            load_frag<kBN, B_RC>(bf, B_RC ? panelB + k : panelB + k * kBN, ldsB, tx);
#pragma unroll
            for (int q = 0; q < 4; ++q)
#pragma unroll
                for (int i = 0; i < 8; ++i) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i][q], bf[j][q], acc[i][j]);
                    if constexpr (EPI == EPI_BWD_W) bsum[i] += a[i][q];
                }
        }
    }
    PPOAF_STAMP(4);

    // epilogue operands (bias / activation of the layer below): their latency hides behind the reduction
    // thread -> row r, columns c4 .. c4+3 (a half-warp reads / writes 256 contiguous bytes)
    const int r = tid >> 4, c4 = (tid & 15) * 4;
    const int m = m0 + r, n = n0 + c4;
    float4 epi = make_float4(0.f, 0.f, 0.f, 0.f);
    if constexpr (EPI == EPI_FWD || EPI == EPI_FWD_DACT) {
        if (n < g.N) epi = load4_guarded(g.bias + n, g.N - n, reinterpret_cast<uintptr_t>(g.bias) % 16 == 0);
    }
    if constexpr (EPI == EPI_BWD_X) {
        if (n < g.N && m < g.M)
            epi = load4_guarded(g.aux + int64_t(m) * g.ldaux + n, g.N - n,
                                g.ldaux % 4 == 0 && reinterpret_cast<uintptr_t>(g.aux) % 16 == 0);
    }

    __syncthreads();                           // panel memory is reused for the split-K reduction
    PPOAF_STAMP(5);

    float* red = smem;                         // [groups][32][72]
    float* red_b = smem + kGroups * kBM * kRedLd;    // [groups][32]
    {   // every group writes (idle groups hold zeros), so the fold below is a fixed, fully unrolled 16-way sum
        float* my = red + (grp * kBM) * kRedLd;
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j)
                my[frag_pos<kBM, A_RC>(ty, i) * kRedLd + frag_pos<kBN, B_RC>(tx, j)] = acc[i][j];
        if constexpr (EPI == EPI_BWD_W) {
            if (tx == 0) {
#pragma unroll
                for (int i = 0; i < 8; ++i) red_b[grp * kBM + frag_pos<kBM, A_RC>(ty, i)] = bsum[i];
            }
        }
    }
    __syncthreads();
    PPOAF_STAMP(6);

    float sq = 0.f;
    float d[4];                                // EPI_FWD_DACT: act'(z) of the four outputs
    if (m < g.M && n < g.N) {
        float4 sum = make_float4(0.f, 0.f, 0.f, 0.f);
        const float* rp = red + r * kRedLd + c4;
#pragma unroll
        for (int gq = 0; gq < kGroups; ++gq) {
            const float4 v = *reinterpret_cast<const float4*>(rp + gq * (kBM * kRedLd));
            sum.x += v.x; sum.y += v.y; sum.z += v.z; sum.w += v.w;
        }
        float o[4] = {sum.x, sum.y, sum.z, sum.w};
        const float e[4] = {epi.x, epi.y, epi.z, epi.w};
        if constexpr (EPI == EPI_FWD) {
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] += e[j];
            act_fwd4<EXT>(o, g.act);
        }
        if constexpr (EPI == EPI_FWD_DACT) {
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float2 yd = act_fwd_grad(o[j] + e[j], g.act);
                o[j] = yd.x; d[j] = yd.y;
            }
        }
        if constexpr (EPI == EPI_BWD_X) act_bwd4<EXT>(o, e, g.act);
        if constexpr (EPI == EPI_BWD_W) {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (n + j < g.N) sq = fmaf(o[j], o[j], sq);
        }
        float* crow = g.C + int64_t(m) * g.ldc;
        if (g.ldc % 4 == 0 && reinterpret_cast<uintptr_t>(g.C) % 16 == 0 && n + 3 < g.N) {
            const float4 o4 = make_float4(o[0], o[1], o[2], o[3]);
            *reinterpret_cast<float4*>(crow + n) = o4;
            if constexpr (EPI == EPI_BWD_W) mirror_store(mir, reinterpret_cast<float4*>(crow + n), o4);
        } else {
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (n + j < g.N) {
                    crow[n + j] = o[j];
                    if constexpr (EPI == EPI_BWD_W) mirror_store(mir, crow + n + j, o[j]);
                }
        }
        if constexpr (EPI == EPI_FWD_DACT) {   // same row pitch as C
            float* drow = g.dact + int64_t(m) * g.ldc;
            if (g.ldc % 4 == 0 && reinterpret_cast<uintptr_t>(g.dact) % 16 == 0 && n + 3 < g.N) {
                *reinterpret_cast<float4*>(drow + n) = make_float4(d[0], d[1], d[2], d[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (n + j < g.N) drow[n + j] = d[j];
            }
        }
        if constexpr (EPI == EPI_BWD_W) {
            if (n0 == 0 && c4 == 0 && g.dbias) {
                float s = 0.f;
#pragma unroll
                for (int gq = 0; gq < kGroups; ++gq) s += red_b[gq * kBM + r];
                g.dbias[m] = s;
                mirror_store(mir, g.dbias + m, s);
                sq = fmaf(s, s, sq);
            }
        }
    }
    PPOAF_STAMP(7);
    if constexpr (EPI == EPI_BWD_W) {
        if (g.sq_out) {                        // per-tile sum of squares -> gradient-norm clip without a norm pass
            __shared__ double s_sq[kThreads / 32];
            const double w = warp_sum(double(sq));
            if (lane == 0) s_sq[grp] = w;
            __syncthreads();
            if (tid == 0) {
                double t = 0.0;
#pragma unroll
                for (int k = 0; k < kThreads / 32; ++k) t += s_sq[k];
                g.sq_out[tile] = t;
            }
        }
    }
}

#ifndef PPOAF_HELPERS_ONLY   // fused_step.cu reuses the helpers above; the kernel itself lives in mlp.cu's translation unit
// Two kernels of one body.  grouped_gemm_kernel takes activation ids 0-3 only; grouped_gemm_ext_kernel takes every id
// and the EPI_FWD_DACT epilogue.  The code of ids 4-11 in the first kernel (one call site per epilogue and four more
// tile instantiations) cost the Tanh C4 benchmark 0.8 % on a B200 at 1000 W, so GemmGroup::launch picks the second
// kernel only for launches that need it.
template <bool EXT>
__device__ __forceinline__ void grouped_gemm_body(const GroupedGemmArgs& args) {
    extern __shared__ __align__(16) float smem[];
    __shared__ __align__(8) uint64_t s_bars[kLoadGroups];
    __shared__ int s_idx[2 * kKRound];
    PPOAF_STAMP(0);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int c = 0; c < kLoadGroups; ++c) mbar_init(&s_bars[c], kThreads);
    }
    __syncthreads();
    int p = 0;
#pragma unroll
    for (int i = 1; i < kMaxGroup; ++i)
        if (i < args.n_problems && int(blockIdx.x) >= args.p[i].tile_begin) p = i;
    const GemmProblem& g = args.p[p];
    const int tile = int(blockIdx.x) - g.tile_begin;
#define PPOAF_TILE(ARC, BRC, VA, VB, E) gemm_tile<ARC, BRC, VA, VB, E, EXT>(g, tile, args.cursor, args.cursor_stride, args.mirror, smem, s_bars, s_idx)
#ifdef PPOAF_GEMM_REPEAT   // debug: run the tile twice, the stamps of the second (warm instruction cache) pass survive
#pragma unroll 1
    for (int rep = 0; rep < 2; ++rep) {
    __syncthreads();
    PPOAF_STAMP(0);
#endif
    switch (g.flavour) {
        case EPI_FWD * 4 + 3: PPOAF_TILE(true, true, 4, 4, EPI_FWD); break;
        case EPI_FWD * 4 + 2: PPOAF_TILE(true, true, 4, 1, EPI_FWD); break;
        case EPI_FWD * 4 + 1: PPOAF_TILE(true, true, 1, 4, EPI_FWD); break;
        case EPI_FWD * 4 + 0: PPOAF_TILE(true, true, 1, 1, EPI_FWD); break;
        case EPI_FWD_DACT * 4 + 3: if constexpr (EXT) { PPOAF_TILE(true, true, 4, 4, EPI_FWD_DACT); } break;
        case EPI_FWD_DACT * 4 + 2: if constexpr (EXT) { PPOAF_TILE(true, true, 4, 1, EPI_FWD_DACT); } break;
        case EPI_FWD_DACT * 4 + 1: if constexpr (EXT) { PPOAF_TILE(true, true, 1, 4, EPI_FWD_DACT); } break;
        case EPI_FWD_DACT * 4 + 0: if constexpr (EXT) { PPOAF_TILE(true, true, 1, 1, EPI_FWD_DACT); } break;
        case EPI_BWD_X * 4 + 3: PPOAF_TILE(true, false, 4, 4, EPI_BWD_X); break;
        case EPI_BWD_X * 4 + 2: PPOAF_TILE(true, false, 4, 1, EPI_BWD_X); break;
        case EPI_BWD_X * 4 + 1: PPOAF_TILE(true, false, 1, 4, EPI_BWD_X); break;
        case EPI_BWD_X * 4 + 0: PPOAF_TILE(true, false, 1, 1, EPI_BWD_X); break;
        case EPI_BWD_W * 4 + 3: PPOAF_TILE(false, false, 4, 4, EPI_BWD_W); break;
        case EPI_BWD_W * 4 + 2: PPOAF_TILE(false, false, 4, 1, EPI_BWD_W); break;
        case EPI_BWD_W * 4 + 1: PPOAF_TILE(false, false, 1, 4, EPI_BWD_W); break;
        default: PPOAF_TILE(false, false, 1, 1, EPI_BWD_W); break;
    }
#ifdef PPOAF_GEMM_REPEAT
    }
#endif
#undef PPOAF_TILE
}
__global__ void __launch_bounds__(kThreads) grouped_gemm_kernel(const GroupedGemmArgs args) { grouped_gemm_body<false>(args); }
__global__ void __launch_bounds__(kThreads) grouped_gemm_ext_kernel(const GroupedGemmArgs args) { grouped_gemm_body<true>(args); }
#endif  // PPOAF_HELPERS_ONLY

}  // namespace ppoaf
