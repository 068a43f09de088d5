// The PPO minibatch step as ONE persistent kernel (reference ppo.py:2292-2468 -> policies/ppo_policy.py:891-952,
// 1012-1055): every minibatch of an epoch runs inside a single launch, one CTA per SM, the phases of a step separated
// by a grid barrier (~0.5 us) instead of a launch boundary (~7 us per dependent launch in the launch-chain path,
// step.cu).  Per step (L = Linear layers per network, actor and critic side by side in every phase):
//
//   FWD l = 0 .. L-2     Y = act(X[idx] W^T + b)                    tcgen05 tiles 128 x bn, 3xTF32
//   LOSS                 the two head layers, PPO loss forward/backward, the heads' dX   (one warp per sample)
//   BWD_X l = L-2 .. 1   dZ_l = (dZ_{l+1} W) * act'(X_l)            tcgen05 tiles 128 x bn
//   BWD_W                dW_l = dZ_{l+1}^T X_l, db_l, per-tile sums of squares (all layers of both networks)
//   ADAM                 gradient-norm clip + Adam on this CTA's slice, counters
//
// GEMM tiles: A (the operand indexed by the 128 tile rows) and B are staged global -> registers -> shared memory
// by 8 warps, which split every fp32 element into hi = tf32(x), lo = tf32(x - hi) on the way (3xTF32:
// D += hi*hi + hi*lo + lo*hi, fp32 accumulation in TMEM, fp32-grade products); a ninth warp issues
// tcgen05.mma (cta_group::1, kind::tf32) from one lane and commits to mbarriers; the 8 warps read the accumulator back
// with tcgen05.ld for the fused epilogues (bias + activation; activation derivative; bias gradient + sum of squares).
// bn (16 / 32 / 64) is chosen per phase so that a phase has about one tile per SM.
// Everything a phase reads that another CTA wrote in an earlier phase is loaded with ld.global.cg (L2), never through L1.
#define PPOAF_HELPERS_ONLY
#include "umma.cuh"
#include "loss_common.cuh"
#include <stdlib.h>
#include <cuda.h>          // CUtensorMap types only: cuTensorMapEncodeTiled is fetched through cudaGetDriverEntryPoint

namespace ppoaf {
namespace fused {

using umma::mbar_init;
using umma::mbar_wait;
using umma::smem_u32;

constexpr int kFM = 128, kFK = 32, kFStages = 4;
constexpr int kStageThreads = 256, kFThreads = kStageThreads + 128;   // 8 staging warps + the MMA warpgroup (warp 8 issues)
constexpr int kStageRegs = 224, kMmaRegs = 56;                        // setmaxnreg: 256 x 224 + 128 x 56 = 168 x 384
constexpr int kMaxBN = 32;
constexpr int kLossSmemFloats = 7168;                                   // head weights + per-warp scratch of the LOSS phase
constexpr int kFTmemCols = 512;
constexpr int kMaxProblems = 6 * PPOAF_MAX_LAYERS;
constexpr int kMaxPhases = 2 * PPOAF_MAX_LAYERS + 2;
constexpr int kBarStride = 8;                                            // one 32-byte sector per CTA arrival word
constexpr int kMaxGrid = 256;

enum { PH_FWD = 0, PH_BWD_X, PH_BWD_W, PH_LOSS, PH_ADAM };

struct PhaseDesc { int type, first, count, n_tiles; };

struct FusedPlan {
    // TMA descriptors of the operands that are plain (un-gathered, 16-byte friendly) matrices: one 2-D box per tile and
    // K chunk (problem flavour bit 4: A through TMA, bit 5: B through TMA); everything else is staged with cp.async
    alignas(64) CUtensorMap tmA[kMaxProblems];
    alignas(64) CUtensorMap tmB[kMaxProblems];
    int n_phases, n_problems, n_steps, batch;
    int loss_finalize_phase;               // phase at whose start the last CTA folds the loss partials
    int batch_size;                        // cursor stride of the permutation
    PhaseDesc ph[kMaxPhases];
    GemmProblem p[kMaxProblems];
    LossArgs loss;
    MirrorSet mirror;
    float* params; const float* grads; float* m; float* v;
    int64_t n_actor, n_total;
    const double* sq_a; int n_sq_a;
    const double* sq_c; int n_sq_c;
    const double* hp;
    int64_t* adam_step;
    int32_t* mb_cursor;
    // gathered minibatch rows, double-buffered by step parity: xg[net] is [2 * batch_size][xg_ld[net]] floats
    float* xg[2]; const float* x_src[2]; int x_dim[2]; int xg_ld[2];
    const int64_t* perm; int64_t n_flat;
    long long* stamps;                     // debug (PPOAF_FUSED_STAMPS=1): clock64 per phase of the last step, CTAs 0 / mid / last
    uint32_t* bar;                         // [0 .. grid*kBarStride): arrival words; [kMaxGrid*kBarStride]: epoch of the last launch
};

__device__ __forceinline__ void st_release_gpu(uint32_t* p, uint32_t v) {
    asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t* p) {
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void bar_stage() { asm volatile("bar.sync 1, %0;" ::"n"(kStageThreads) : "memory"); }

// Grid barrier (all CTAs are co-resident: cooperative launch, one CTA per SM).  CTA b publishes `epoch` in its own
// arrival word; the threads of CTA 0 each poll one arrival word and CTA 0 then releases a single "go" word that one
// thread of every other CTA polls: two L2 round trips after the last arrival, no contended atomic, and (unlike every CTA
// polling every word, measured: 175 MB of L2 reads per step) almost no polling traffic competing with the operand loads.
__device__ __forceinline__ void grid_sync(uint32_t* arrive, uint32_t epoch) {
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) {
        // flat counter: every CTA adds one and polls the same word until it reads epoch * grid (the grid size is the same
        // for every launch on a workspace, so the count carries over from launch to launch like the epoch does).  One L2
        // round trip shorter than an arrival word per CTA gathered by CTA 0 + a release word (measured: 5.5K -> 2.5K clk)
        uint32_t* cnt = arrive + kMaxGrid * kBarStride + 4;
        const uint32_t target = epoch * gridDim.x;
        asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(cnt) : "memory");
        while (int32_t(ld_acquire_gpu(cnt) - target) < 0) {}
    }
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// 4 consecutive floats (zero beyond n_valid) straight from L2
__device__ __forceinline__ float4 ldcg4(const float* __restrict__ p, int n_valid, bool vec) {
    if (n_valid <= 0) return make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec && n_valid >= 4) return __ldcg(reinterpret_cast<const float4*>(p));
    float4 v;
    v.x = __ldcg(p);
    v.y = n_valid > 1 ? __ldcg(p + 1) : 0.f;
    v.z = n_valid > 2 ? __ldcg(p + 2) : 0.f;
    v.w = n_valid > 3 ? __ldcg(p + 3) : 0.f;
    return v;
}

// =========================================================================================================
// GEMM tile pipeline.  Per 32-wide K chunk and pipeline stage s:
//   producer warp   : TMA bulk copies (cp.async.bulk, one per operand row) global -> raw fp32 tiles in shared memory,
//                     completion counted in bytes on raw_full[s]                                     (warp 9)
//   converter warps : raw tile -> hi = tf32(x), lo = tf32(x - hi);  A (128 tile rows = 128 TMEM lanes, 32 k = 32 + 32
//                     columns) goes to TENSOR MEMORY with tcgen05.st, B goes to shared memory in the UMMA layout;
//                     arrive on op_full[s] and raw_free[s]                                            (warps 0..7)
//   MMA issuer      : tcgen05.mma kind::tf32 with A from TMEM (TS mode), 3 MMAs per k-step of 8
//                     (hi*hi -> "big" accumulator, hi*lo + lo*hi -> "small" accumulator); tcgen05.commit frees stage s
//                     on mma_free[s]                                                                   (warp 8, one lane)
// A from TMEM: with 16-column tiles an SS-mode MMA re-reads 4 KB of A from shared memory per 16 K MACs and the tile is
// bound by the 128 B/clk shared-memory port (measured); TMEM feeds the tensor core without touching it.
// Accuracy: the tensor core accumulates with truncation, so a single fp32 accumulator over K = 512 is ~10x less accurate
// than an fp32 FMA chain.  Chunks are therefore dealt round-robin over kParts accumulator pairs (big / small terms
// apart) that the epilogue adds in fp32 round-to-nearest: fp32-FMA-grade results (emulated and measured).
// Operands that are not 16-byte friendly (ld or extent not a multiple of 4 floats: first layers of 18 / 54 inputs, the
// head gradients) skip the raw tile: the converters read them from global memory directly.
// =========================================================================================================
constexpr int kRawLdA = 32;                                   // raw K-major rows are dense (128 B) with their 16-byte chunks XOR-swizzled by
                                                              // (row & 7): the layout TMA SWIZZLE_128B writes, conflict-free for the
                                                              // converters' one-row-per-lane LDS.128
constexpr int kRawAFloats = kFM * kRawLdA;                    // 16 KB (MN-major raw A: 32 x 128 floats, unswizzled)
constexpr int kRawBFloats = kMaxBN * kRawLdA;                 // 4 KB  (MN-major raw B: 32 x bn floats)
constexpr int kOpBFloats = kMaxBN * kFK;                      // one UMMA B tile (hi or lo)
constexpr int kRawStages = 6;                                  // raw (TMA / cp.async) ring: deeper than the operand ring, the L2 -> shared
                                                              // memory latency under 148 CTAs' load is ~2.4K clk (measured), several chunks
constexpr int kRawStageFloats = kRawAFloats + kRawBFloats;    // 20 KB
constexpr int kOpStageFloats = 2 * kOpBFloats;                // B hi | lo in the UMMA layout (A hi | lo live in TMEM), kFStages of them
constexpr int kParts = 4;                                     // accumulator pairs
static_assert((kRawAFloats * 4) % 1024 == 0 && (kRawStageFloats * 4) % 1024 == 0 && (kOpStageFloats * 4) % 1024 == 0, "stage layout");
constexpr int kTileSmemFloats = kRawStages * kRawStageFloats + kFStages * kOpStageFloats;
constexpr size_t kFusedSmemBytes = (size_t(kTileSmemFloats) + kLossSmemFloats) * sizeof(float) + 1024;
constexpr int kTmemA = 0, kTmemAcc = 256;                     // TMEM columns: A stages 4 x (32 hi | 32 lo), accumulators 8 x 32

__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void bulk_g2s(float* smem_dst, const float* gsrc, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
// Executed by ALL lanes of the MMA warp with warp-uniform operands; one elected lane issues.  (Issuing from inside an
// `if (lane == 0)` branch makes the compiler wrap every UTCHMMA in an ELECT / R2UR.BROADCAST / BRA.U.ANY waterfall, ~85 clk
// per instruction: measured.)
__device__ __forceinline__ void mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p, q;\n\telect.sync _|q, 0xffffffff;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}\n" ::"r"(tmem_d), "r"(tmem_a), "l"(db), "r"(idesc),
        "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit_elect(uint64_t* bar) {
    asm volatile(
        "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
        "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}\n" ::"r"(smem_u32(bar))
        : "memory");
}
// tf32 round-to-nearest (ties away) with integer arithmetic: add half an ulp of the 10-bit mantissa, clear the 13 low bits.
// Same result as cvt.rna.tf32.f32 for finite normal inputs, but IADD + LOP run at 64 lanes/clk/SM whereas the conversion
// unit runs at 16: with cvt the split was ~600 of the ~1100 clk a converter warp spends per K chunk (measured).
__device__ __forceinline__ float tf32_round(float x) {
    return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xFFFFE000u);
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const float (&v)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};\n" ::"r"(taddr),
        "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])), "r"(__float_as_uint(v[3])),
        "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])), "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])),
        "r"(__float_as_uint(v[8])), "r"(__float_as_uint(v[9])), "r"(__float_as_uint(v[10])), "r"(__float_as_uint(v[11])),
        "r"(__float_as_uint(v[12])), "r"(__float_as_uint(v[13])), "r"(__float_as_uint(v[14])), "r"(__float_as_uint(v[15]))
        : "memory");
}
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
}

struct TileBars {            // raw_*: [kRawStages]; op_full / mma_free: [kFStages]
    uint64_t* raw_full; uint64_t* raw_free; uint64_t* op_full; uint64_t* mma_free; uint64_t* acc;
};
__device__ __forceinline__ float* stage_raw_a(float* smem, int sr) { return smem + sr * kRawStageFloats; }
__device__ __forceinline__ float* stage_raw_b(float* smem, int sr) { return smem + sr * kRawStageFloats + kRawAFloats; }
__device__ __forceinline__ float* stage_op_b(float* smem, int s) { return smem + kRawStages * kRawStageFloats + s * kOpStageFloats; }

// whether an operand travels through a raw tile (TMA bulk copies need 16-byte aligned rows and sizes)
__device__ __forceinline__ bool a_is_raw(const GemmProblem& g) { return (g.flavour & 2) != 0; }
__device__ __forceinline__ bool b_is_raw(const GemmProblem& g) { return (g.flavour & 1) != 0; }

// ---- producers (warps 9..11, 96 threads): cp.async of both operand tiles of a chunk into the raw stage ----
// 16-byte copies when the operand is 16-byte friendly (flavour bits), 4-byte copies otherwise; rows / columns beyond the
// operand's extent are zero-filled (src-size 0), so the raw tiles are always fully defined.
constexpr int kProdThreads = 128;          // warps 8..11: each produces (cp.async / TMA) AND issues one k-step's MMAs
constexpr int kLook = kRawStages - 1;        // chunks the producer side runs ahead of the MMA side inside a tile
// KROWS: the tile rows are reduction indices (MN-major raw tile): rows beyond the extent must be ZERO (they are multiplied into
// valid outputs) while columns beyond the extent only feed outputs that are never stored and are skipped; K-major tiles
// (KROWS = false) the other way round.  row_add: address-only row offset (odd-step half of a double-buffered operand).
template <bool VEC, bool SWZ, bool KROWS>
__device__ __forceinline__ void copy_tile(float* dst, int dst_ld, const float* __restrict__ P, int ld, const int64_t* __restrict__ idx,
                                          int row0, int n_rows, int row_ext, int col0, int n_cols, int col_ext, int row_add, int pt) {
    const int nr = KROWS ? n_rows : min(n_rows, row_ext - row0);
    int nc = KROWS ? min(n_cols, col_ext - col0) : n_cols;
    if (nr <= 0 || nc <= 0) return;
    if constexpr (VEC) {
        int cpr = 1;                                          // 16-byte chunks per row, rounded up to a power of two
        while (cpr * 4 < nc) cpr <<= 1;
        const int sh = 31 - __clz(cpr);
        for (int op = pt; op < nr * cpr; op += kProdThreads) {
            const int r = op >> sh, c4 = op & (cpr - 1);
            const bool ok = row0 + r < row_ext && col0 + 4 * c4 < col_ext;
            const int64_t gr = ok ? (idx ? idx[row0 + r] : int64_t(row0 + r + row_add)) : 0;
            const int pc = SWZ ? (c4 ^ (r & 7)) : c4;
            cp_async_16(dst + r * dst_ld + 4 * pc, P + gr * ld + (ok ? col0 + 4 * c4 : 0), ok);
        }
    } else {
        int ncp = 1;
        while (ncp < nc) ncp <<= 1;
        const int sh = 31 - __clz(ncp);
        for (int op = pt; op < nr * ncp; op += kProdThreads) {
            const int r = op >> sh, c = op & (ncp - 1);
            const bool ok = row0 + r < row_ext && col0 + c < col_ext;
            const int64_t gr = ok ? (idx ? idx[row0 + r] : int64_t(row0 + r + row_add)) : 0;
            const int pc = SWZ ? ((((c >> 2) ^ (r & 7)) << 2) | (c & 3)) : c;
            cp_async_4(dst + r * dst_ld + pc, P + gr * ld + (ok ? col0 + c : 0), ok);
        }
    }
}

__device__ __forceinline__ void mbar_expect_tx_only(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_2d(float* smem_dst, const CUtensorMap* tm, int c0, int c1, uint64_t* bar) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(tm)), "r"(c0), "r"(c1), "r"(smem_u32(bar))
                 : "memory");
}

// One K chunk of both operand tiles -> raw stage (executed by the 128 threads of the MMA warpgroup).
template <bool A_RC, bool B_RC>
__device__ __forceinline__ void produce_chunk(const GemmProblem& g, const CUtensorMap* tmA, const CUtensorMap* tmB, int m0, int n0,
                                              const int64_t* idxA, const int64_t* idxB, int addA, int addB, int c, uint32_t gc,
                                              float* smem, const TileBars& tb) {
    const int pt = int(threadIdx.x) - kStageThreads;
    const int bn = g.bn;
    const bool vecA = (g.flavour & 2) != 0, vecB = (g.flavour & 1) != 0;
    const bool tmaA = (g.flavour & 16) != 0, tmaB = (g.flavour & 32) != 0;
    const uint32_t tma_bytes = (tmaA ? uint32_t(kFM * kFK * 4) : 0u) + (tmaB ? uint32_t(bn * kFK * 4) : 0u);   // whole boxes (OOB = zeros)
    const int s = int(gc % kRawStages);
    const int k0 = c * kFK;
    if (gc >= uint32_t(kRawStages)) mbar_wait(&tb.raw_free[s], (gc / kRawStages - 1u) & 1u);
    float* ra = stage_raw_a(smem, s);
    float* rb = stage_raw_b(smem, s);
    if (pt == 0 && tma_bytes) {
        // one TMA box per operand: K-major {k0, row0} -> [rows][32] swizzled; MN-major {out0, k0} -> [32][outs]
        mbar_expect_tx_only(&tb.raw_full[s], tma_bytes);
        if (tmaA) { if constexpr (A_RC) tma_load_2d(ra, tmA, k0, m0 + addA, &tb.raw_full[s]); else tma_load_2d(ra, tmA, m0, k0 + addA, &tb.raw_full[s]); }
        if (tmaB) { if constexpr (B_RC) tma_load_2d(rb, tmB, k0, n0 + addB, &tb.raw_full[s]); else tma_load_2d(rb, tmB, n0, k0 + addB, &tb.raw_full[s]); }
    }
    if (!tmaA) {
        if constexpr (A_RC) {      // raw A[r = tile row][k]:  A[row(m0 + r) * lda + k0 + k]
            if (vecA) copy_tile<true, true, false>(ra, kRawLdA, g.A, g.lda, idxA, m0, kFM, g.M, k0, kFK, g.K, addA, pt);
            else copy_tile<false, true, false>(ra, kRawLdA, g.A, g.lda, idxA, m0, kFM, g.M, k0, kFK, g.K, addA, pt);
        } else {                   // raw A[k][m = tile row]:  A[row(k0 + k) * lda + m0 + m]
            if (vecA) copy_tile<true, false, true>(ra, kFM, g.A, g.lda, idxA, k0, kFK, g.K, m0, kFM, g.M, addA, pt);
            else copy_tile<false, false, true>(ra, kFM, g.A, g.lda, idxA, k0, kFK, g.K, m0, kFM, g.M, addA, pt);
        }
    }
    if (!tmaB) {
        if constexpr (B_RC) {
            if (vecB) copy_tile<true, true, false>(rb, kRawLdA, g.B, g.ldb, idxB, n0, bn, g.N, k0, kFK, g.K, addB, pt);
            else copy_tile<false, true, false>(rb, kRawLdA, g.B, g.ldb, idxB, n0, bn, g.N, k0, kFK, g.K, addB, pt);
        } else {
            if (vecB) copy_tile<true, false, true>(rb, bn, g.B, g.ldb, idxB, k0, kFK, g.K, n0, bn, g.N, addB, pt);
            else copy_tile<false, false, true>(rb, bn, g.B, g.ldb, idxB, k0, kFK, g.K, n0, bn, g.N, addB, pt);
        }
    }
    cp_async_arrive(&tb.raw_full[s]);                     // one arrival per thread once its copies (if any) have landed
}

// ---- MMA warpgroup (warps 8..11): producer AND issuer ----
// A tcgen05.mma costs ~80-100 clk of issue whatever its shape (measured), so the four k-steps of a chunk are split over the
// four warps (`ks` = warp - 8: disjoint accumulators, every warp commits to the stage / accumulator barriers).  The same
// warps feed the pipeline: before issuing chunk c they put chunk c + kLook in flight (TMA box loads by one thread, cp.async
// by all 128 for operands TMA cannot describe), so the loads run kLook chunks ahead of the MMAs inside a tile.
template <bool A_RC, bool B_RC>
__device__ __forceinline__ void ftile_mma(const GemmProblem& g, const CUtensorMap* tmA, const CUtensorMap* tmB, int tile,
                                          int64_t idx_off, int odd, uint32_t ks, float* smem, const TileBars& tb, uint32_t tmem,
                                          uint32_t& gchunk, long long* dbg) {
    const int bn = g.bn;
    const int m0 = (tile / g.tiles_n) * kFM, n0 = (tile % g.tiles_n) * bn;
    const int n_chunks = (g.K + kFK - 1) / kFK;
    const uint32_t c0 = gchunk;
    gchunk += uint32_t(n_chunks);
    const int64_t* idxA = g.idxA ? g.idxA + idx_off : nullptr;
    const int64_t* idxB = g.idxB ? g.idxB + idx_off : nullptr;
    const int addA = odd ? g.a_par : 0, addB = odd ? g.b_par : 0;
    // A comes from TMEM (K-major by construction); B from shared memory
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((B_RC ? 0u : 1u) << 16) | (uint32_t(bn >> 3) << 17) |
                           (uint32_t(kFM >> 4) << 24);
    const uint64_t db0 = umma::desc_base<B_RC>();
    const uint64_t ob = ks * umma::kstep_units<B_RC>();
    uint32_t d0, d1, d2;
    // every (k-step, term) owns its accumulator, so consecutive MMAs are independent
    // (12 slots of 16 columns; at bn = 32 the two small terms of a k-step share one: 8 slots of 32 columns)
    if (bn == 16) { d0 = tmem + uint32_t(kTmemAcc) + (ks * 3u) * 16u; d1 = d0 + 16u; d2 = d0 + 32u; }
    else { d0 = tmem + uint32_t(kTmemAcc) + (ks * 2u) * 32u; d1 = d0 + 32u; d2 = d1; }
    for (int c = 0; c < kLook && c < n_chunks; ++c)
        produce_chunk<A_RC, B_RC>(g, tmA, tmB, m0, n0, idxA, idxB, addA, addB, c, c0 + uint32_t(c), smem, tb);
    for (int c = 0; c < n_chunks; ++c) {
        if (c + kLook < n_chunks)
            produce_chunk<A_RC, B_RC>(g, tmA, tmB, m0, n0, idxA, idxB, addA, addB, c + kLook, c0 + uint32_t(c + kLook), smem, tb);
        const uint32_t gc = c0 + uint32_t(c);
        const int s = int(gc % kFStages);
        if (dbg && c < 8) dbg[3 * c] = clock64();
        mbar_wait(&tb.op_full[s], (gc / kFStages) & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (dbg && c < 8) dbg[3 * c + 1] = clock64();
        const uint32_t sb = smem_u32(stage_op_b(smem, s));
        const uint64_t b_hi = db0 | uint64_t((sb >> 4) & 0x3FFF);
        const uint64_t b_lo = db0 | uint64_t(((sb + kOpBFloats * 4) >> 4) & 0x3FFF);
        const uint32_t a_hi = tmem + uint32_t(kTmemA + s * 64), a_lo = a_hi + 32u;
        const bool first = c == 0;                            // first chunk: overwrite
        mma_tf32_ts(d0, a_hi + 8u * ks, b_hi + ob, idesc, first ? 0u : 1u);
        mma_tf32_ts(d1, a_hi + 8u * ks, b_lo + ob, idesc, first ? 0u : 1u);
        mma_tf32_ts(d2, a_lo + 8u * ks, b_hi + ob, idesc, (first && bn == 16) ? 0u : 1u);
        umma_commit_elect(&tb.mma_free[s]);
        if (dbg && c < 8) dbg[3 * c + 2] = clock64();
    }
    umma_commit_elect(tb.acc);
}

// ---- converters + epilogue (warps 0..7) ----
template <bool A_RC, bool B_RC, int EPI>
__device__ __forceinline__ void ftile(const GemmProblem& g, int tile, int64_t idx_off, const MirrorSet& mir, float* smem,
                                      const TileBars& tb, uint32_t tmem, uint32_t& gchunk, uint32_t& gtile, double* s_sq,
                                      long long* dbg) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int bn = g.bn;
    if (dbg) dbg[0] = clock64();
    const int m0 = (tile / g.tiles_n) * kFM, n0 = (tile % g.tiles_n) * bn;
    const int n_chunks = (g.K + kFK - 1) / kFK;
    const uint32_t c0 = gchunk, acc_parity = gtile & 1u;
    gchunk += uint32_t(n_chunks);
    gtile += 1u;
    const int q = warp & 3, h = warp >> 2;                    // TMEM lane group / k half of the chunk (A), column half (epilogue)
    const int ml = q * 32 + lane;                             // this thread's tile row (= TMEM lane)
    const int m = m0 + ml;

    // The converters work as two groups of four warps (one warp per TMEM lane quarter): group `h` takes the chunks whose
    // global index has parity h, so the two groups' wait -> LDS -> split -> tcgen05.st -> fence -> arrive chains overlap.
    // B quads of this thread: 4 consecutive floats of the contiguous direction, bn * 8 quads per chunk over 128 threads
    const int gt = tid & 127;
    const int gpr = B_RC ? 8 : (bn >> 2);                     // quads per raw row
    const int n_bq = bn * 8;
    int b_src[2], b_dst[2];
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        const int t = gt + 128 * j;
        const int b_r = t / gpr, b_g = t % gpr;               // K-major: (row n, k quad);  MN-major: (k row, output quad)
        if constexpr (B_RC) {
            b_src[j] = b_r * kRawLdA + ((b_g ^ (b_r & 7)) << 2);
            b_dst[j] = b_r * 32 + ((b_g ^ (b_r & 7)) * 4);
        } else {
            b_src[j] = b_r * bn + 4 * b_g;
            b_dst[j] = (b_g / 8) * 1024 + (b_r / 4) * 128 + (b_r % 4) * 32 + ((((b_g / 2) % 4) ^ (b_r % 4)) * 8) + (b_g % 2) * 4;
        }
    }
    float rowsum = 0.f;                                       // EPI_BWD_W: bias gradient = sum over k of this thread's A row

    // epilogue operands are fetched now, so their latency hides behind the main loop
    const int half = bn >> 1;                                 // columns per warp: 8 or 16
    const int nb = n0 + h * half;
    const bool vec_out = (g.ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(g.C) % 16 == 0);
    float4 epi[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        epi[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int n = nb + 4 * j;
        if (4 * j < half) {
            if constexpr (EPI == EPI_FWD) {
                if (n < g.N) epi[j] = ldcg4(g.bias + n, g.N - n, vec_out);
            }
            if constexpr (EPI == EPI_BWD_X) {
                if (n < g.N && m < g.M) epi[j] = ldcg4(g.aux + int64_t(m) * g.ldaux + n, g.N - n, vec_out && g.ldaux % 4 == 0);
            }
        }
    }
    if (dbg) dbg[1] = clock64();

#pragma unroll 1
    for (int c = int((c0 ^ uint32_t(h)) & 1u); c < n_chunks; c += 2) {
        const uint32_t gc = c0 + uint32_t(c);
        const int s = int(gc % kFStages), sr = int(gc % kRawStages);
        float x[32];
        float4 bq[2];
        bq[0] = bq[1] = make_float4(0.f, 0.f, 0.f, 0.f);
        mbar_wait(&tb.raw_full[sr], (gc / kRawStages) & 1u);
        if (dbg && c < 12) dbg[4 + 2 * c] = clock64();
        {
            const float* ra = stage_raw_a(smem, sr);
            if constexpr (A_RC) {
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const float4 v = *reinterpret_cast<const float4*>(ra + ml * kRawLdA + ((i ^ (ml & 7)) << 2));
                    x[4 * i] = v.x; x[4 * i + 1] = v.y; x[4 * i + 2] = v.z; x[4 * i + 3] = v.w;
                }
            } else {
#pragma unroll
                for (int i = 0; i < 32; ++i) x[i] = ra[i * kFM + ml];
            }
        }
        {
            const float* rb = stage_raw_b(smem, sr);
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (gt + 128 * j < n_bq) bq[j] = *reinterpret_cast<const float4*>(rb + b_src[j]);
        }
        // the raw tile may be refilled as soon as every warp of the group has read it
        __syncwarp();
        if (lane == 0) mbar_arrive(&tb.raw_free[sr]);
        if (dbg && c == 4) dbg[29] = clock64();

        float4 bh[2], bl[2];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            bh[j].x = tf32_round(bq[j].x); bl[j].x = tf32_round(bq[j].x - bh[j].x);
            bh[j].y = tf32_round(bq[j].y); bl[j].y = tf32_round(bq[j].y - bh[j].y);
            bh[j].z = tf32_round(bq[j].z); bl[j].z = tf32_round(bq[j].z - bh[j].z);
            bh[j].w = tf32_round(bq[j].w); bl[j].w = tf32_round(bq[j].w - bh[j].w);
        }
        // the MMAs of chunk gc - kFStages have finished reading this stage's TMEM columns and B tiles
        if (dbg && c == 4) dbg[30] = clock64();
        if (gc >= uint32_t(kFStages)) mbar_wait(&tb.mma_free[s], (gc / kFStages - 1u) & 1u);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        if (dbg && c == 4) dbg[31] = clock64();
        const uint32_t ta = tmem + (uint32_t(q * 32) << 16) + uint32_t(kTmemA + s * 64);
#pragma unroll
        for (int kh = 0; kh < 2; ++kh) {
            float hi[16], lo[16];
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const float v = x[16 * kh + i];
                hi[i] = tf32_round(v);
                lo[i] = tf32_round(v - hi[i]);
                if constexpr (EPI == EPI_BWD_W) rowsum += v;
            }
            tmem_st16(ta + uint32_t(16 * kh), hi);
            tmem_st16(ta + 32u + uint32_t(16 * kh), lo);
        }
        {
            float* ob = stage_op_b(smem, s);
#pragma unroll
            for (int j = 0; j < 2; ++j)
                if (gt + 128 * j < n_bq) {
                    *reinterpret_cast<float4*>(ob + b_dst[j]) = bh[j];
                    *reinterpret_cast<float4*>(ob + kOpBFloats + b_dst[j]) = bl[j];
                }
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        if (dbg && c == 4) dbg[26] = clock64();
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
        if (dbg && c == 4) dbg[27] = clock64();
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) mbar_arrive(&tb.op_full[s]);
        if (dbg && c < 12) dbg[5 + 2 * c] = clock64();
    }
    if (dbg) dbg[2] = clock64();
    mbar_wait(tb.acc, acc_parity);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if (dbg) dbg[3] = clock64();

    // ---- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31, columns half (w / 4) .. +half-1 of every accumulator in
    // use, 8 columns at a time; small terms first, then the big ones, fp32 round-to-nearest ----
    const int n_slots = bn == 16 ? 12 : 8;
    float sq = 0.f;
    float* crow = g.C + int64_t(m) * g.ldc;
    const int act = g.act;
#pragma unroll
    for (int j8 = 0; j8 < kMaxBN / 2; j8 += 8) {
        if (j8 >= half) break;                      // warp-uniform
        float v8[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) v8[j] = 0.f;
        const uint32_t tcol = tmem + (uint32_t(q * 32) << 16) + uint32_t(kTmemAcc + h * half + j8);
        // every accumulator slot in flight at once (one TMEM round trip instead of twelve), then the sums in a fixed
        // order: small-term accumulators first, the big ones last
        uint32_t r[12][8];
#pragma unroll
        for (int sl = 0; sl < 12; ++sl) {
            if (sl < n_slots) tmem_ld8(tcol + uint32_t(sl * bn), r[sl]);
            else {
#pragma unroll
                for (int j = 0; j < 8; ++j) r[sl][j] = 0u;
            }
        }
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (dbg && j8 == 0) dbg[20] = clock64();
#pragma unroll
        for (int pass = 0; pass < 2; ++pass) {
#pragma unroll
            for (int sl = 0; sl < 12; ++sl) {
                const bool small = bn == 16 ? (sl % 3 != 0) : (sl % 2 == 1);
                if (small == (pass == 0)) {
#pragma unroll
                    for (int j = 0; j < 8; ++j) v8[j] += __uint_as_float(r[sl][j]);
                }
            }
        }
        if (dbg && j8 == 0) dbg[21] = clock64();
        if (m < g.M) {
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
                const int n = nb + j8 + 4 * jj;
                const float4 e4 = epi[(j8 >> 2) + jj];
                const float ev[4] = {e4.x, e4.y, e4.z, e4.w};
                float o[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v = v8[4 * jj + j];
                    if constexpr (EPI == EPI_FWD) v = act_fwd_fast(v + ev[j], act);
                    if constexpr (EPI == EPI_BWD_X) v *= act_bwd_from_out(ev[j], act);
                    if constexpr (EPI == EPI_BWD_W) { if (n + j < g.N) sq = fmaf(v, v, sq); }
                    o[j] = v;
                }
                if (vec_out && n + 3 < g.N) {
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
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");   // the next tile's MMAs overwrite the accumulators
    if (dbg) dbg[28] = clock64();

    if constexpr (EPI == EPI_BWD_W) {
        // bias gradient: this thread summed its row over the chunks of its group; the two groups meet in shared memory
        __shared__ float s_rowsum[2][kFM];
        s_rowsum[h][ml] = rowsum;
        const double w = warp_sum(double(sq));
        bar_stage();
        float db = 0.f;
        if (tid < kFM) {
            db = s_rowsum[0][tid] + s_rowsum[1][tid];
            if (n0 == 0 && g.dbias && m0 + tid < g.M) {
                g.dbias[m0 + tid] = db;
                mirror_store(mir, g.dbias + m0 + tid, db);
            }
        }
        const double wdb = warp_sum((n0 == 0 && tid < kFM && m0 + tid < g.M) ? double(db) * double(db) : 0.0);
        if (lane == 0) s_sq[warp] = w + wdb;
        bar_stage();
        if (tid == 0 && g.sq_out) {
            double t = 0.0;
#pragma unroll
            for (int k = 0; k < kStageThreads / 32; ++k) t += s_sq[k];
            g.sq_out[tile] = t;
        }
        bar_stage();                                 // s_rowsum / s_sq are reused by the next tile
    }
}

static_assert(kLossThreads == kStageThreads, "the staging warps run the shared loss code (loss_common.cuh)");
struct StageBarrier { __device__ __forceinline__ void operator()() const { bar_stage(); } };

// Head weights of both networks -> shared memory.  They were written by the ADAM phase of the previous step (several grid
// barriers ago), so the staging warps run this BEFORE the grid barrier that opens the LOSS phase: the L2 loads overlap the
// wait for the slowest CTA of the last hidden layer.
__device__ __forceinline__ void loss_stage_heads(const LossArgs& a, float* s_dyn, float* s_sd, float* s_dsd) {
    const int tid = threadIdx.x;
    const HeadSmem hs(a, s_dyn);
    const int qa = a.Ha / 4;
    for (int t = tid; t < hs.prows * qa; t += kStageThreads) {
        const int row = t / qa, c4 = t - row * qa;
        const float4 w = row < a.pred_dim ? __ldcg(reinterpret_cast<const float4*>(a.W_actor + int64_t(row) * a.Ha + 4 * c4))
                                          : make_float4(0.f, 0.f, 0.f, 0.f);
        *reinterpret_cast<float4*>(hs.wa + row * hs.ldw + 4 * c4) = w;
    }
    for (int t = tid; t < a.Hc / 4; t += kStageThreads)
        *reinterpret_cast<float4*>(hs.wc + 4 * t) = __ldcg(reinterpret_cast<const float4*>(a.W_critic + 4 * t));
    if (tid < a.pred_dim) hs.b[tid] = __ldcg(a.b_actor + tid);
    if (tid == 0) hs.b[a.pred_dim] = __ldcg(a.b_critic);
    if (a.head == PPOAF_HEAD_GAUSSIAN_TANH && tid < a.act_dim) s_sd[tid] = std_of_log_std(__ldcg(a.log_std + tid), a.min_std, s_dsd[tid]);
}

// ---------------------------------------------------------------------------------------------------------
// LOSS phase: one warp per sample, samples dealt round-robin over CTAs so that every SM holds 3-4 of a 512-row
// minibatch.  Head layers, loss and the heads' dX as in ppo_loss_kernel<true> (loss.cu); the per-CTA partial sums are
// folded by the last CTA at the start of the next phase (loss_finalize).
__device__ __forceinline__ void loss_phase(const LossArgs& a, int cur, float* s_dyn, float* s_sd, double (*s_red)[kPartialStride],
                                           long long* dbg) {
    if (dbg) dbg[0] = clock64();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gl = lane;
    const float inv_b = 1.0f / float(a.batch);
    const float w_ent = float(a.hparams[PPOAF_HP_ENTROPY_WEIGHT]);
    const float clip_lo = float(1.0 - a.hparams[PPOAF_HP_SURR_CLIP]), clip_hi = float(1.0 + a.hparams[PPOAF_HP_SURR_CLIP]);
    const bool gaussian = a.head == PPOAF_HEAD_GAUSSIAN_TANH;
    const HeadSmem hs(a, s_dyn);

    float adv_mu = 0.f, adv_sd = 1.f, val_mu = 0.f, val_sd = 1.f;    // this minibatch's normalisation constants
    if (a.normalize_adv) { adv_mu = a.mb_adv_stats[2 * cur]; adv_sd = a.mb_adv_stats[2 * cur + 1]; }
    if (a.normalize_values) { val_mu = a.mb_val_stats[2 * cur]; val_sd = a.mb_val_stats[2 * cur + 1]; }
    const int64_t* idx = a.perm + int64_t(cur) * a.batch_size;
    bar_stage();
    if (dbg) dbg[1] = clock64();

    double tot_sc[kLossScalars];
    double tot_dsd[kPerLane];
#pragma unroll
    for (int k = 0; k < kLossScalars; ++k) tot_sc[k] = 0.0;
#pragma unroll
    for (int k = 0; k < kPerLane; ++k) tot_dsd[k] = 0.0;

    for (int i = warp * int(gridDim.x) + int(blockIdx.x); i < a.batch; i += (kStageThreads / 32) * int(gridDim.x)) {
        const int64_t j = idx[i];
        const int64_t nxt = int64_t(cur + 1) * a.batch_size + i;
        const int64_t jn = (a.pf_rows[0] && nxt < a.n_flat) ? a.perm[nxt] : -1;
        float adv = a.advantages[j];
        const float lp_old = a.log_probs[j];
        float target = a.rewards_to_go[j];
        float4 ha[kFusedMaxChunks], hc[kFusedMaxChunks];
        const float* hra = a.h_actor + int64_t(i) * a.Ha + 4 * gl;
        const float* hrc = a.h_critic + int64_t(i) * a.Hc + 4 * gl;
#pragma unroll
        for (int c = 0; c < kFusedMaxChunks; ++c) {
            const int col = 4 * (gl + kG * c);
            ha[c] = col < a.Ha ? __ldcg(reinterpret_cast<const float4*>(hra + 4 * kG * c)) : make_float4(0.f, 0.f, 0.f, 0.f);
            hc[c] = col < a.Hc ? __ldcg(reinterpret_cast<const float4*>(hrc + 4 * kG * c)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (jn >= 0) {   // pull the NEXT minibatch's observation rows into L2 while this step's backward pass runs
            const char* r0 = reinterpret_cast<const char*>(a.pf_rows[0]) + jn * a.pf_row_bytes[0];
            const char* r1 = reinterpret_cast<const char*>(a.pf_rows[1]) + jn * a.pf_row_bytes[1];
            for (int o = gl * 128; o < a.pf_row_bytes[0]; o += kG * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r0 + o));
            for (int o = gl * 128; o < a.pf_row_bytes[1]; o += kG * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(r1 + o));
        }
        float sc[kLossScalars];
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) sc[k] = 0.f;
        float dsd[kPerLane];
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) dsd[k] = 0.f;
        if (a.normalize_adv) adv = (adv - adv_mu) / adv_sd;
        if (a.normalize_values) target = (target - val_mu) / val_sd;
        if (dbg) dbg[2] = clock64();

        const float v = head_forward(a, hs, ha, hc, gl, hs.pred + warp * kFusedPredLd);
        if (dbg) dbg[3] = clock64();
        if (gl == 0) a.values[j] = v;                                 // dataset.values[batch_idxs] = values (ppo.py:2340)
        float bad_value = isnan(v) ? 1.f : 0.f;

        const float* pred = hs.pred + warp * kFusedPredLd;
        float* dpred = a.d_actor_out + int64_t(i) * (a.d_actor_ld ? a.d_actor_ld : a.pred_dim);
        float* sdp = hs.dpred + warp * kFusedPredLd;
        actor_head_loss<true>(a, a.head, true, gl, j, pred, dpred, sdp, s_sd, adv, lp_old, inv_b, w_ent, clip_lo, clip_hi, sc,
                              dsd, bad_value);

        if (dbg) dbg[4] = clock64();
        // ---- critic ----
        float dv1 = 0.f;
        sc[LS_CRITIC] = critic_term(v, target, a.use_huber, dv1);
        if (gl != 0) sc[LS_CRITIC] = 0.f;
        if (gl == 0) a.d_critic_out[int64_t(i) * (a.d_critic_ld ? a.d_critic_ld : 1)] = dv1 * inv_b;
        const float bad_any = group_max(bad_value);
        sc[LS_BAD_VALUE] = gl == 0 ? bad_any : 0.f;

        head_backward(a, hs, ha, hc, sdp, dv1, inv_b, true, gl, i);
        __syncwarp();                                                // s_pred / s_dpred are reused by the next sample
        if (dbg) dbg[5] = clock64();
#pragma unroll
        for (int k = 0; k < kLossScalars; ++k) tot_sc[k] += double(sc[k]);
#pragma unroll
        for (int k = 0; k < kPerLane; ++k) tot_dsd[k] += double(dsd[k]);
    }

    loss_cta_partials(tot_sc, tot_dsd, kLossScalars + (gaussian ? a.act_dim : 0), s_red, reinterpret_cast<double*>(a.partials),
                      StageBarrier{});
    bar_stage();
    if (dbg) dbg[6] = clock64();
}

// Totals of the loss partials -> d(log_std) (+ its sum of squares) and the epoch statistics.  Run by the staging warps
// of the last CTA at the start of the phase after LOSS (the partials are visible after the grid barrier).  The fused
// engine never clips values (loss_head_fusable), so the critic loss is the unclipped one.
__device__ __forceinline__ void loss_finalize(const LossArgs& a, const float* s_dsd, double (*s_red)[kPartialStride],
                                              double* s_tot, double* s_sq) {
    const float w_ent = float(a.hparams[PPOAF_HP_ENTROPY_WEIGHT]);
    loss_fold(a, kLossScalars + (a.head == PPOAF_HEAD_GAUSSIAN_TANH ? a.act_dim : 0), s_dsd, s_red, s_tot, s_sq,
              StageBarrier{});
    if (threadIdx.x == 0) add_epoch_stats(a, s_tot, float(s_tot[LS_CRITIC] / double(a.batch)), w_ent);
    bar_stage();
}

// ---------------------------------------------------------------------------------------------------------
// ADAM phase: arithmetic of adam_update_kernel (optim.cu) on this CTA's slice; t, beta^t are carried in registers /
// shared memory across the steps of the launch.
struct AdamC { float neg_step_size, bc2_sqrt, w1, beta2, w2, eps, inv_world; };
__device__ __forceinline__ void adam_vec4(float4& pq, const float4& gq, float4& mq, float4& vq, float coef, const AdamC& c) {
    float g[4] = {gq.x, gq.y, gq.z, gq.w}, p[4] = {pq.x, pq.y, pq.z, pq.w};
    float mm[4] = {mq.x, mq.y, mq.z, mq.w}, vv[4] = {vq.x, vq.y, vq.z, vq.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const float gk = __fmul_rn(__fmul_rn(g[k], c.inv_world), coef);
        mm[k] = __fadd_rn(mm[k], __fmul_rn(c.w1, __fsub_rn(gk, mm[k])));
        vv[k] = __fadd_rn(__fmul_rn(vv[k], c.beta2), __fmul_rn(__fmul_rn(c.w2, gk), gk));
        float sq;                                      // approximate sqrt / divisions: same arithmetic as optim.cu (adam_vec)
        asm("sqrt.approx.f32 %0, %1;" : "=f"(sq) : "f"(vv[k]));
        const float denom = __fadd_rn(__fdividef(sq, c.bc2_sqrt), c.eps);
        p[k] = __fadd_rn(p[k], __fdividef(__fmul_rn(c.neg_step_size, mm[k]), denom));
    }
    pq = make_float4(p[0], p[1], p[2], p[3]);
    mq = make_float4(mm[0], mm[1], mm[2], mm[3]);
    vq = make_float4(vv[0], vv[1], vv[2], vv[3]);
}

__device__ __forceinline__ void adam_phase(const FusedPlan& P, double p1, double p2, double* s_scr, float* s_f, long long* dbg) {
    if (dbg) dbg[0] = clock64();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int64_t nv = P.n_total / 4, na = P.n_actor / 4;
    const int64_t stride = int64_t(gridDim.x) * kStageThreads;
    const int64_t i0 = int64_t(blockIdx.x) * kStageThreads + tid;
    float4* p4 = reinterpret_cast<float4*>(P.params);
    const float4* g4 = reinterpret_cast<const float4*>(P.grads);
    float4* m4 = reinterpret_cast<float4*>(P.m);
    float4* v4 = reinterpret_cast<float4*>(P.v);
    constexpr int kSlots = 4;
    float4 G[kSlots], Pq[kSlots], M[kSlots], V[kSlots];
#pragma unroll
    for (int k = 0; k < kSlots; ++k) {
        const int64_t i = i0 + k * stride;
        if (i < nv) { G[k] = __ldcg(g4 + i); Pq[k] = __ldcg(p4 + i); M[k] = __ldcg(m4 + i); V[k] = __ldcg(v4 + i); }
    }
    // fold the sum-of-squares slots (same order in every CTA -> identical scalars everywhere)
    double ta = 0.0, tc = 0.0;
    for (int k = tid; k < P.n_sq_a; k += kStageThreads) ta += __ldcg(P.sq_a + k);
    for (int k = tid; k < P.n_sq_c; k += kStageThreads) tc += __ldcg(P.sq_c + k);
    if (dbg) dbg[1] = clock64();
    ta = warp_sum(ta);
    tc = warp_sum(tc);
    if (lane == 0) { s_scr[warp] = ta; s_scr[8 + warp] = tc; }
    bar_stage();
    if (dbg) dbg[2] = clock64();
    if (tid == 0) {
        double sa = 0.0, sc = 0.0;
#pragma unroll
        for (int k = 0; k < kStageThreads / 32; ++k) { sa += s_scr[k]; sc += s_scr[8 + k]; }
        const double* hp = P.hp;
        const float inv_world = float(hp[PPOAF_HP_INV_WORLD]);
        const float max_norm = float(hp[PPOAF_HP_GRAD_CLIP]);
        const double scale = double(inv_world);
        const float ca = clip_coef(max_norm, sa, scale), cc = clip_coef(max_norm, sc, scale);
        const double b1d = hp[PPOAF_HP_BETA1], b2d = hp[PPOAF_HP_BETA2];
        const double bc1 = 1.0 - p1, bc2 = 1.0 - p2;
        s_f[0] = float(-(hp[PPOAF_HP_LR] / bc1));
        s_f[1] = float(sqrt(bc2));
        s_f[2] = float(1.0 - b1d);
        s_f[3] = float(b2d);
        s_f[4] = float(1.0 - b2d);
        s_f[5] = float(hp[PPOAF_HP_ADAM_EPS]);
        s_f[6] = inv_world;
        s_f[7] = ca;
        s_f[8] = cc;
    }
    bar_stage();
    if (dbg) dbg[3] = clock64();
    const AdamC c{s_f[0], s_f[1], s_f[2], s_f[3], s_f[4], s_f[5], s_f[6]};
    const float coef_a = s_f[7], coef_c = s_f[8];
#pragma unroll
    for (int k = 0; k < kSlots; ++k) {
        const int64_t i = i0 + k * stride;
        if (i < nv) {
            adam_vec4(Pq[k], G[k], M[k], V[k], i < na ? coef_a : coef_c, c);
            p4[i] = Pq[k]; m4[i] = M[k]; v4[i] = V[k];
        }
    }
    for (int64_t i = i0 + kSlots * stride; i < nv; i += stride) {
        const float4 gq = __ldcg(g4 + i);
        float4 pq = __ldcg(p4 + i), mq = __ldcg(m4 + i), vq = __ldcg(v4 + i);
        adam_vec4(pq, gq, mq, vq, i < na ? coef_a : coef_c, c);
        p4[i] = pq; m4[i] = mq; v4[i] = vq;
    }
    if (dbg) { dbg[4] = clock64(); dbg[5] = (long long)__float_as_int(Pq[0].x); }
    bar_stage();                                                    // s_scr / s_f are reused by the next step
    if (dbg) dbg[6] = clock64();
}

// Rows of minibatch `mb` (perm[mb * B + r]) of both observation arrays -> the contiguous half `odd` of xg: the first-layer
// GEMMs (forward and dW) then read a plain matrix through TMA instead of gathering 16 bytes at a time.  Rows beyond the
// minibatch's extent are zero-filled (they are reduction rows of the first-layer dW).  All converter threads of all CTAs.
__device__ __forceinline__ void gather_minibatch(const FusedPlan& P, int mb, int odd) {
    const int B = P.batch_size;
    const int64_t first = int64_t(mb) * B;
    const int64_t left = P.n_flat - first;
    const int rows = int(left < 0 ? 0 : (left < B ? left : B));
    const int tid = threadIdx.x;
    for (int r = int(blockIdx.x); r < B; r += int(gridDim.x)) {
        const int64_t j = r < rows ? P.perm[first + r] : -1;
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int D = P.x_dim[k], ld = P.xg_ld[k];
            float* dst = P.xg[k] + (size_t(odd) * B + r) * ld;
            const float* src = P.x_src[k] + (j < 0 ? 0 : j) * D;
            if ((D & 3) == 0 && (reinterpret_cast<uintptr_t>(P.x_src[k]) & 15) == 0) {
                for (int c = tid; c < D / 4; c += kStageThreads) {
                    const float4 v = j >= 0 ? ldg_stream_f4(reinterpret_cast<const float4*>(src) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
                    reinterpret_cast<float4*>(dst)[c] = v;
                }
            } else {
                for (int c = tid; c < ld; c += kStageThreads) dst[c] = (j >= 0 && c < D) ? src[c] : 0.f;
            }
        }
    }
}

__global__ void __launch_bounds__(kFThreads, 1) ppo_fused_step_kernel(const __grid_constant__ FusedPlan P) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t s_bars[2 * kRawStages + 2 * kFStages + 1];
    __shared__ uint32_t s_tmem;
    __shared__ float s_sd[kMaxAct], s_dsd[kMaxAct];
    __shared__ double s_red[kStageThreads / 32][kPartialStride];
    __shared__ double s_tot[kPartialStride];
    __shared__ double s_sq[kStageThreads / 32];
    __shared__ double s_scr[16];
    __shared__ float s_f[12];
    float* smem = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, warp = tid >> 5;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kFTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 32) {
#pragma unroll
        for (int i = 0; i < kRawStages; ++i) {
            mbar_init(&s_bars[i], kProdThreads);                   // raw_full: one cp.async arrival per thread of the MMA warpgroup
            mbar_init(&s_bars[kRawStages + i], kStageThreads / 64);   // raw_free: one arrival per warp of the converter group that owns the chunk
        }
#pragma unroll
        for (int i = 0; i < kFStages; ++i) {
            mbar_init(&s_bars[2 * kRawStages + i], kStageThreads / 64);          // op_full: likewise
            mbar_init(&s_bars[2 * kRawStages + kFStages + i], 4);                // mma_free: one tcgen05.commit per issuer warp
        }
        mbar_init(&s_bars[2 * kRawStages + 2 * kFStages], 4);      // accumulators complete (all four issuers)
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = __shfl_sync(0xffffffffu, s_tmem, 0);
    const TileBars tb{s_bars, s_bars + kRawStages, s_bars + 2 * kRawStages, s_bars + 2 * kRawStages + kFStages, s_bars + 2 * kRawStages + 2 * kFStages};
    float* loss_smem = smem + kTileSmemFloats;

    // launch-wide state, read before the first grid barrier (the counters are only written at the very end)
    uint32_t epoch = P.bar[kMaxGrid * kBarStride];
    const int cur0 = *P.mb_cursor;
    const int64_t t0 = *P.adam_step;

    if (warp >= kStageThreads / 32) {
        // ============================ MMA warpgroup: warp 8 / lane 0 issues, the rest only keeps the barriers company ============================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kMmaRegs));
        uint32_t gchunk = 0;
        const uint32_t ks = uint32_t(warp - kStageThreads / 32);   // this warp's k-step of every chunk
        for (int step = 0; step < P.n_steps; ++step) {
            const int64_t idx_off = int64_t(cur0 + step) * P.batch_size;
            for (int ph = 0; ph < P.n_phases; ++ph) {
                grid_sync(P.bar, ++epoch);                        // (before the very first phase: the gathered rows of step 0)
                const PhaseDesc d = P.ph[ph];
                if (d.type == PH_LOSS || d.type == PH_ADAM) continue;
                if (tid == kStageThreads) asm volatile("fence.proxy.async;" ::: "memory");   // other CTAs' generic-proxy writes -> TMA reads
                for (int t = int(blockIdx.x); t < d.n_tiles; t += int(gridDim.x)) {
                    int pi = d.first;
                    for (int i = d.first + 1; i < d.first + d.count; ++i)
                        if (t >= P.p[i].tile_begin) pi = i;
                    long long* mdbg = (P.stamps && blockIdx.x == 0 && t == 0 && step == P.n_steps - 1 && tid == kStageThreads)
                                          ? P.stamps + 3 * kMaxPhases * 4 + kMaxPhases * 32 + ph * 32 : nullptr;
                    const int tile = t - P.p[pi].tile_begin;
                    if (d.type == PH_FWD) ftile_mma<true, true>(P.p[pi], &P.tmA[pi], &P.tmB[pi], tile, idx_off, step & 1, ks, smem, tb, tmem, gchunk, mdbg);
                    else if (d.type == PH_BWD_X) ftile_mma<true, false>(P.p[pi], &P.tmA[pi], &P.tmB[pi], tile, idx_off, step & 1, ks, smem, tb, tmem, gchunk, mdbg);
                    else ftile_mma<false, false>(P.p[pi], &P.tmA[pi], &P.tmB[pi], tile, idx_off, step & 1, ks, smem, tb, tmem, gchunk, mdbg);
                }
            }
        }
    } else {
        // ============================ staging / epilogue / loss / optimizer warps ============================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kStageRegs));
        double p1 = 0.0, p2 = 0.0;
        const double b1d = P.hp[PPOAF_HP_BETA1], b2d = P.hp[PPOAF_HP_BETA2];
        if (tid == 0) { p1 = pow(b1d, double(t0)); p2 = pow(b2d, double(t0)); }
        uint32_t gchunk = 0, gtile = 0;
        gather_minibatch(P, cur0, 0);                                  // step 0's rows; later steps are gathered in the LOSS phase
        for (int step = 0; step < P.n_steps; ++step) {
            const int cur = cur0 + step;
            const int64_t idx_off = int64_t(cur) * P.batch_size;
            p1 *= b1d; p2 *= b2d;                                     // beta^t of this step (thread 0)
            for (int ph = 0; ph < P.n_phases; ++ph) {
                long long* stp = nullptr;
                if (P.stamps && tid == 0 && step == P.n_steps - 1) {
                    const int slot = blockIdx.x == 0 ? 0 : (blockIdx.x == gridDim.x / 2 ? 1 : (blockIdx.x == gridDim.x - 1 ? 2 : -1));
                    if (slot >= 0) stp = P.stamps + (slot * kMaxPhases + ph) * 4;
                }
                if (stp) stp[0] = clock64();
                const PhaseDesc d = P.ph[ph];
                if (d.type == PH_LOSS) loss_stage_heads(P.loss, loss_smem, s_sd, s_dsd);
                grid_sync(P.bar, ++epoch);
                if (stp) stp[1] = clock64();
                if (ph == P.loss_finalize_phase && blockIdx.x == gridDim.x - 1) loss_finalize(P.loss, s_dsd, s_red, s_tot, s_sq);
                if (d.type == PH_LOSS) {
                    loss_phase(P.loss, cur, loss_smem, s_sd, s_red, (stp && blockIdx.x == 0) ? P.stamps + 3 * kMaxPhases * 4 + ph * 32 : nullptr);
                    if (step + 1 < P.n_steps) gather_minibatch(P, cur + 1, (step + 1) & 1);   // read again 4 barriers from now
                } else if (d.type == PH_ADAM) {
                    adam_phase(P, p1, p2, s_scr, s_f, (stp && blockIdx.x == 0) ? P.stamps + 3 * kMaxPhases * 4 + ph * 32 : nullptr);
                } else {
                    for (int t = int(blockIdx.x); t < d.n_tiles; t += int(gridDim.x)) {
                        int pi = d.first;
                        for (int i = d.first + 1; i < d.first + d.count; ++i)
                            if (t >= P.p[i].tile_begin) pi = i;
                        const GemmProblem& g = P.p[pi];
                        long long* tdbg = (stp && blockIdx.x == 0 && t == 0) ? P.stamps + 3 * kMaxPhases * 4 + ph * 32 : nullptr;
                        const int tile = t - g.tile_begin;
                        if (d.type == PH_FWD) ftile<true, true, EPI_FWD>(g, tile, idx_off, P.mirror, smem, tb, tmem, gchunk, gtile, s_sq, tdbg);
                        else if (d.type == PH_BWD_X) ftile<true, false, EPI_BWD_X>(g, tile, idx_off, P.mirror, smem, tb, tmem, gchunk, gtile, s_sq, tdbg);
                        else ftile<false, false, EPI_BWD_W>(g, tile, idx_off, P.mirror, smem, tb, tmem, gchunk, gtile, s_sq, tdbg);
                    }
                }
                if (stp) stp[2] = clock64();
            }
        }
        // counters of the launch: every CTA read them before its first grid barrier
        if (blockIdx.x == 0 && tid == 0) {
            *P.adam_step = t0 + P.n_steps;
            *P.mb_cursor = cur0 + P.n_steps;
            P.bar[kMaxGrid * kBarStride] = epoch;
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kFTmemCols));
}

}  // namespace fused
}  // namespace ppoaf

// =========================================================================================================
// host side: workspace layout, plan construction, entry points
// =========================================================================================================
namespace ppoaf {
namespace fused {

struct FScratch {
    uint32_t* bar;
    double* sq_actor; double* sq_critic;
    int n_sq_actor, n_sq_critic;
    double* loss_partials;
    float* act[2][PPOAF_MAX_LAYERS + 1];
    float* dz[2][PPOAF_MAX_LAYERS + 1];
    float* xg[2];                 // gathered minibatch rows, [2 * max_batch][xg_ld]
    int xg_ld[2];
    size_t total;
};

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }
static int max_w_tiles(const ppoaf_mlp_desc* net) {      // upper bound of the backward-w tiles of one network (bn = 32)
    int n = 0;
    for (int l = 0; l < net->n_layers; ++l) n += ceil_div(net->dims[l + 1], kFM) * ceil_div(net->dims[l], 32);
    return n;
}

static void fcarve(const ppoaf_update_cfg* cfg, int max_batch, char* base, FScratch* out) {
    size_t off = 0;
    auto take = [&](size_t bytes) {
        char* p = base ? base + off : nullptr;
        off += align_up(bytes, 256);
        return p;
    };
    // control words first, at offsets that do not depend on the batch: they persist from launch to launch
    out->bar = reinterpret_cast<uint32_t*>(take(sizeof(uint32_t) * (size_t(kMaxGrid) * kBarStride + 8)));
    out->n_sq_actor = max_w_tiles(&cfg->actor) + 1;
    out->n_sq_critic = max_w_tiles(&cfg->critic);
    out->sq_actor = reinterpret_cast<double*>(take(size_t(out->n_sq_actor) * sizeof(double)));
    out->sq_critic = reinterpret_cast<double*>(take(size_t(out->n_sq_critic) * sizeof(double)));
    out->loss_partials = reinterpret_cast<double*>(take(size_t(kMaxGrid) * kPartialStride * sizeof(double)));
    const ppoaf_mlp_desc* nets[2] = {&cfg->actor, &cfg->critic};
    for (int k = 0; k < 2; ++k)
        for (int l = 1; l <= nets[k]->n_layers; ++l) {
            out->act[k][l] = reinterpret_cast<float*>(take(size_t(max_batch) * nets[k]->dims[l] * sizeof(float)));
            out->dz[k][l] = reinterpret_cast<float*>(take(size_t(max_batch) * ((nets[k]->dims[l] + 3) / 4 * 4) * sizeof(float)));
        }
    for (int k = 0; k < 2; ++k) {
        out->xg_ld[k] = (nets[k]->dims[0] + 3) / 4 * 4;          // 16-byte row pitch: TMA-able whatever the observation width
        out->xg[k] = reinterpret_cast<float*>(take(size_t(2) * max_batch * out->xg_ld[k] * sizeof(float)));
    }
    out->total = off;
}

static const char* unsupported_reason(const ppoaf_update_cfg* cfg) {
    const int La = cfg->actor.n_layers, Lc = cfg->critic.n_layers;
    if (La != Lc) return "actor and critic depths differ";
    if (La < 2) return "networks without a hidden layer";
    if (cfg->actor.activation != cfg->critic.activation) return "actor and critic activations differ";
    if (!loss_head_fusable(cfg->actor.dims[La], cfg->actor.dims[La - 1], cfg->critic.dims[Lc - 1], cfg->vf_clip_enabled))
        return "head layers are not fusable (hidden width > 256 or not a multiple of 4, > 24 actor outputs, or value clipping)";
    if (cfg->act_dim > kMaxAct || cfg->actor.dims[La] > kMaxAct) return "action width out of range";
    if (cfg->world_size > 1) return "multi-rank exchange runs through the launch-chain path";
    return nullptr;
}

// ---- TMA descriptors (driver entry point fetched at run time: the library links cudart only) ----
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        const char* e = getenv("PPOAF_FUSED_TMA");
        if (e && e[0] == '0') return nullptr;                     // PPOAF_FUSED_TMA=0: cp.async for every operand
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
        else
            (void)cudaGetLastError();
    }
    return fn;
}
// matrix [n_rows x n_cols] fp32, row stride ld floats; box = box_cols (contiguous) x box_rows; K-major raw tiles take the
// 128-byte swizzle (box_cols = 32), MN-major raw tiles are plain
static bool make_tmap(CUtensorMap* tm, const float* base, int64_t n_rows, int64_t n_cols, int64_t ld, int box_cols, int box_rows,
                      bool swizzle128) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn || reinterpret_cast<uintptr_t>(base) % 16 != 0 || (ld * 4) % 16 != 0 || box_cols > 256 || box_rows > 256) return false;
    const cuuint64_t gdim[2] = {cuuint64_t(n_cols), cuuint64_t(n_rows)};
    const cuuint64_t gstride[1] = {cuuint64_t(ld) * 4};
    const cuuint32_t box[2] = {cuuint32_t(box_cols), cuuint32_t(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    const CUresult r = fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                          CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                          CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS;
}

static inline bool vec4_ok(const float* p, int ld, int contig_extent) {
    return (reinterpret_cast<uintptr_t>(p) % 16 == 0) && (ld % 4 == 0) && (contig_extent % 4 == 0);
}

// tile width of a phase: the widest bn whose tile count reaches ~2/3 of the grid, else the narrowest allowed
static int pick_bn(int grid, int min_bn, const int (*MN)[2], int n_prob) {
    const int cand[2] = {32, 16};
    for (int c = 0; c < 2; ++c) {
        const int bn = cand[c];
        if (bn < min_bn) break;
        int tiles = 0;
        for (int i = 0; i < n_prob; ++i) tiles += ceil_div(MN[i][0], kFM) * ceil_div(MN[i][1], bn);
        if (tiles * 3 >= grid * 2 || bn == min_bn) return bn;
    }
    return min_bn;
}

static int build_plan(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* b, int n_steps, int grid, FusedPlan* P) {
    memset(P, 0, sizeof(*P));
    FScratch sc;
    fcarve(cfg, b->batch_size, reinterpret_cast<char*>(b->workspace), &sc);
    const bool gaussian = cfg->head == PPOAF_HEAD_GAUSSIAN_TANH;
    int64_t off[2][2 * PPOAF_MAX_LAYERS + 1];
    const int64_t n_actor = param_layout(&cfg->actor, gaussian ? cfg->act_dim : 0, off[0]);
    const int64_t n_critic = param_layout(&cfg->critic, 0, off[1]);
    const ppoaf_mlp_desc* net[2] = {&cfg->actor, &cfg->critic};
    const float* par[2] = {b->params, b->params + n_actor};
    float* grd[2] = {b->grads, b->grads + n_actor};
    const float* x0[2] = {b->obs, b->critic_obs};
    const int L = cfg->actor.n_layers;
    const int rows = b->batch;

    P->n_steps = n_steps;
    P->batch = rows;
    P->batch_size = b->batch_size;
    int np = 0, nph = 0;
    auto begin_phase = [&](int type) { P->ph[nph].type = type; P->ph[nph].first = np; P->ph[nph].count = 0; P->ph[nph].n_tiles = 0; };
    auto add_problem = [&](GemmProblem& g, int bn) {
        g.bn = bn;
        // operands that are plain 16-byte-friendly matrices travel through TMA (no gather: a tensor map cannot indirect)
        const int epi = g.flavour >> 2;
        const bool a_rc = epi != EPI_BWD_W, b_rc = epi == EPI_FWD;
        if (!g.idxA) {
            // K-major A: matrix [M x K] (ld = lda), box 32 x 128;  MN-major A (dZ as [K x M]): box 128 x 32.  An operand
            // that alternates between two halves by step parity is described as ONE matrix of both halves (a_par rows apart)
            const bool ok = a_rc ? make_tmap(&P->tmA[np], g.A, g.M + g.a_par, g.K, g.lda, kFK, kFM, true)
                                 : make_tmap(&P->tmA[np], g.A, g.K + g.a_par, g.M, g.lda, kFM, kFK, false);
            if (ok) g.flavour |= 16;
        }
        if (!g.idxB) {
            const bool ok = b_rc ? make_tmap(&P->tmB[np], g.B, g.N + g.b_par, g.K, g.ldb, kFK, bn, true)
                                 : make_tmap(&P->tmB[np], g.B, g.K + g.b_par, g.N, g.ldb, bn, kFK, false);
            if (ok) g.flavour |= 32;
        }
        g.tiles_n = ceil_div(g.N, bn);
        g.tile_begin = P->ph[nph].n_tiles;
        P->ph[nph].n_tiles += g.tiles_n * ceil_div(g.M, kFM);
        P->ph[nph].count += 1;
        P->p[np++] = g;
    };

    // ---- forward, hidden layers ----
    for (int l = 0; l < L - 1; ++l) {
        begin_phase(PH_FWD);
        const int MN[2][2] = {{rows, net[0]->dims[l + 1]}, {rows, net[1]->dims[l + 1]}};
        const int bn = pick_bn(grid, 16, MN, 2);
        for (int k = 0; k < 2; ++k) {
            GemmProblem g{};
            const float* X = l == 0 ? sc.xg[k] : sc.act[k][l];
            const int in = net[k]->dims[l], out = net[k]->dims[l + 1];
            const int ldx = l == 0 ? sc.xg_ld[k] : in;
            const float* W = par[k] + off[k][2 * l];
            g.A = X; g.lda = ldx; g.B = W; g.ldb = in; g.C = sc.act[k][l + 1]; g.ldc = out;
            g.M = rows; g.N = out; g.K = in;
            g.a_par = l == 0 ? b->batch_size : 0;
            g.bias = par[k] + off[k][2 * l + 1];
            g.act = net[k]->activation;
            g.flavour = EPI_FWD * 4 + (vec4_ok(X, ldx, in) ? 2 : 0) + (vec4_ok(W, in, in) ? 1 : 0);
            add_problem(g, bn);
        }
        ++nph;
    }
    // ---- heads + loss ----
    begin_phase(PH_LOSS);
    ++nph;
    P->loss_finalize_phase = nph;
    // ---- backward-x, top hidden layer first ----
    for (int l = L - 2; l >= 1; --l) {
        begin_phase(PH_BWD_X);
        const int MN[2][2] = {{rows, net[0]->dims[l]}, {rows, net[1]->dims[l]}};
        const int bn = pick_bn(grid, 32, MN, 2);          // MN-major B tiles: groups of 32 outputs
        for (int k = 0; k < 2; ++k) {
            GemmProblem g{};
            const int in = net[k]->dims[l], out = net[k]->dims[l + 1];
            const float* W = par[k] + off[k][2 * l];
            g.A = sc.dz[k][l + 1]; g.lda = out; g.B = W; g.ldb = in; g.C = sc.dz[k][l]; g.ldc = in;
            g.M = rows; g.N = in; g.K = out;
            g.aux = sc.act[k][l]; g.ldaux = in; g.act = net[k]->activation;
            g.flavour = EPI_BWD_X * 4 + (vec4_ok(g.A, out, out) ? 2 : 0) + (vec4_ok(W, in, in) ? 1 : 0);
            add_problem(g, bn);
        }
        ++nph;
    }
    // ---- backward-w, every layer of both networks in one phase ----
    {
        begin_phase(PH_BWD_W);
        int MN[2 * PPOAF_MAX_LAYERS][2];
        int cnt = 0;
        for (int k = 0; k < 2; ++k)
            for (int l = 0; l < L; ++l) { MN[cnt][0] = net[k]->dims[l + 1]; MN[cnt][1] = net[k]->dims[l]; ++cnt; }
        const int bn = pick_bn(grid, 32, MN, cnt);
        double* sq[2] = {sc.sq_actor, sc.sq_critic};
        int used[2] = {0, 0};
        for (int k = 0; k < 2; ++k)
            for (int l = L - 1; l >= 0; --l) {             // widest-K problems (none here: K = rows for all) / top layers first
                GemmProblem g{};
                const int in = net[k]->dims[l], out = net[k]->dims[l + 1];
                const float* X = l == 0 ? sc.xg[k] : sc.act[k][l];
                const int ldx = l == 0 ? sc.xg_ld[k] : in;
                const int lddz = l == L - 1 ? (out + 3) / 4 * 4 : out;      // the head gradients are stored with a 16-byte row pitch
                g.A = sc.dz[k][l + 1]; g.lda = lddz; g.B = X; g.ldb = ldx; g.C = grd[k] + off[k][2 * l]; g.ldc = in;
                g.M = out; g.N = in; g.K = rows;
                g.b_par = l == 0 ? b->batch_size : 0;
                g.dbias = grd[k] + off[k][2 * l + 1];
                g.sq_out = sq[k] + used[k];
                g.flavour = EPI_BWD_W * 4 + (vec4_ok(g.A, lddz, out) ? 2 : 0) + (vec4_ok(X, ldx, in) ? 1 : 0);
                used[k] += ceil_div(out, kFM) * ceil_div(in, bn);
                add_problem(g, bn);
            }
        P->sq_a = sc.sq_actor; P->n_sq_a = used[0] + 1;     // + the log_std slot (zero for the Categorical head)
        P->sq_c = sc.sq_critic; P->n_sq_c = used[1];
        ++nph;
    }
    begin_phase(PH_ADAM);
    ++nph;
    P->n_phases = nph;
    P->n_problems = np;

    // ---- loss arguments (fused heads) ----
    LossArgs& a = P->loss;
    a.log_std = gaussian ? par[0] + off[0][2 * L] : nullptr;
    a.raw_actions = b->raw_actions;
    a.advantages = b->advantages;
    a.log_probs = b->log_probs;
    a.rewards_to_go = b->rewards_to_go;
    a.values = b->values;
    a.perm = b->perm;
    a.cursor = b->mb_cursor;
    a.batch_size = b->batch_size;
    a.batch = rows;
    a.mb_adv_stats = b->mb_adv_stats;
    a.mb_val_stats = b->mb_val_stats;
    a.hparams = b->hparams;
    a.epoch_stats = b->epoch_stats;
    a.d_actor_out = sc.dz[0][L];
    a.d_critic_out = sc.dz[1][L];
    a.d_actor_ld = (cfg->actor.dims[L] + 3) / 4 * 4;
    a.d_critic_ld = 4;
    a.d_log_std = gaussian ? grd[0] + off[0][2 * L] : nullptr;
    a.sq_log_std = sc.sq_actor + (P->n_sq_a - 1);
    a.partials = reinterpret_cast<float*>(sc.loss_partials);
    a.head = cfg->head;
    a.act_dim = cfg->act_dim;
    a.pred_dim = cfg->actor.dims[L];
    a.section_ends = cfg_section_ends(cfg);
    a.use_huber = cfg->use_huber;
    a.normalize_adv = cfg->normalize_adv;
    a.normalize_values = cfg->normalize_values;
    a.vf_clip_enabled = 0;
    a.min_std = cfg->min_std;
    a.pf_rows[0] = nullptr;                 // the next minibatch's rows are GATHERED during the LOSS phase instead of prefetched
    a.pf_rows[1] = nullptr;
    a.pf_row_bytes[0] = cfg->actor.dims[0] * int(sizeof(float));
    a.pf_row_bytes[1] = cfg->critic.dims[0] * int(sizeof(float));
    a.n_flat = b->n_flat;
    a.n_mirror = 0;
    a.fused = 1;
    a.h_actor = sc.act[0][L - 1];
    a.h_critic = sc.act[1][L - 1];
    a.W_actor = par[0] + off[0][2 * (L - 1)];
    a.b_actor = par[0] + off[0][2 * (L - 1) + 1];
    a.W_critic = par[1] + off[1][2 * (L - 1)];
    a.b_critic = par[1] + off[1][2 * (L - 1) + 1];
    a.dz_actor = sc.dz[0][L - 1];
    a.dz_critic = sc.dz[1][L - 1];
    a.Ha = cfg->actor.dims[L - 1];
    a.Hc = cfg->critic.dims[L - 1];
    a.act = cfg->actor.activation;

    for (int k = 0; k < 2; ++k) {
        P->xg[k] = sc.xg[k]; P->xg_ld[k] = sc.xg_ld[k]; P->x_src[k] = x0[k]; P->x_dim[k] = net[k]->dims[0];
    }
    P->perm = b->perm;
    P->n_flat = b->n_flat;
    P->mirror.n = 0;
    P->params = b->params; P->grads = b->grads; P->m = b->adam_m; P->v = b->adam_v;
    P->n_actor = n_actor; P->n_total = n_actor + n_critic;
    P->hp = b->hparams;
    P->adam_step = b->adam_step;
    P->mb_cursor = b->mb_cursor;
    P->bar = sc.bar;
    return 0;
}

static long long* g_stamps = nullptr;
static long long* stamp_buffer() {          // debug only
    static int enabled = -1;
    if (enabled < 0) { const char* e = getenv("PPOAF_FUSED_STAMPS"); enabled = (e && e[0] == '1') ? 1 : 0; }
    if (!enabled) return nullptr;
    if (!g_stamps) {
        if (cudaMalloc(&g_stamps, sizeof(long long) * (3 * kMaxPhases * 4 + 2 * kMaxPhases * 32)) != cudaSuccess) { g_stamps = nullptr; return nullptr; }
        cudaMemset(g_stamps, 0, sizeof(long long) * (3 * kMaxPhases * 4 + 2 * kMaxPhases * 32));
    }
    return g_stamps;
}

static bool g_fused_configured = false;
static void configure_fused() {
    g_fused_configured = true;
    cudaFuncSetAttribute(ppo_fused_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(kFusedSmemBytes));
}

}  // namespace fused
}  // namespace ppoaf

using namespace ppoaf;

extern "C" int ppoaf_ppo_fused_supported(const ppoaf_update_cfg* cfg) {
    if (!cfg) return 0;
    if (check_mlp_desc(&cfg->actor, "ppoaf_ppo_fused_supported") || check_mlp_desc(&cfg->critic, "ppoaf_ppo_fused_supported")) return 0;
    const char* why = fused::unsupported_reason(cfg);
    if (why) { set_error("ppoaf_ppo_fused_steps: not supported: %s", why); return 0; }
    return 1;
}

extern "C" size_t ppoaf_ppo_fused_workspace_bytes(const ppoaf_update_cfg* cfg, int32_t max_batch) {
    if (!cfg || max_batch <= 0) return 0;
    fused::FScratch s;
    fused::fcarve(cfg, max_batch, nullptr, &s);
    return s.total;
}

extern "C" int ppoaf_ppo_fused_steps(const ppoaf_update_cfg* cfg, const ppoaf_update_bufs* b, int32_t n_steps, void* stream) {
    PPOAF_CHECK_ARG(cfg != nullptr && b != nullptr, "ppoaf_ppo_fused_steps: null argument");
    if (check_cfg(cfg, "ppoaf_ppo_fused_steps")) return 1;
    const char* why = fused::unsupported_reason(cfg);
    PPOAF_CHECK_ARG(why == nullptr, "ppoaf_ppo_fused_steps: not supported: %s", why ? why : "");
    PPOAF_CHECK_ARG(b->batch >= 2 && b->batch <= b->batch_size && b->n_flat > 0 && n_steps >= 1,
                    "ppoaf_ppo_fused_steps: bad batch sizes (one-row minibatches are skipped by the caller)");
    PPOAF_CHECK_ARG(n_steps == 1 || b->batch == b->batch_size, "ppoaf_ppo_fused_steps: several steps need full minibatches");
    PPOAF_CHECK_ARG(b->workspace_bytes >= ppoaf_ppo_fused_workspace_bytes(cfg, b->batch_size),
                    "ppoaf_ppo_fused_steps: workspace too small");
    PPOAF_CHECK_ARG(reinterpret_cast<uintptr_t>(b->workspace) % 256 == 0, "ppoaf_ppo_fused_steps: workspace must be 256-byte aligned");
    PPOAF_CHECK_ARG((cfg->actor.n_layers * 6) <= fused::kMaxProblems, "ppoaf_ppo_fused_steps: too many layers");
    if (!fused::g_fused_configured) fused::configure_fused();
    int grid = sm_count();
    if (grid > fused::kMaxGrid) grid = fused::kMaxGrid;
    static thread_local fused::FusedPlan plan;
    if (fused::build_plan(cfg, b, n_steps, grid, &plan)) return 1;
    plan.stamps = fused::stamp_buffer();

    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3(grid); lc.blockDim = dim3(fused::kFThreads); lc.dynamicSmemBytes = fused::kFusedSmemBytes;
    lc.stream = (cudaStream_t)stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative;      // all CTAs co-resident: the phases are separated by grid barriers
    attr[0].val.cooperative = 1;
    lc.attrs = attr; lc.numAttrs = 1;
    cudaError_t e = cudaLaunchKernelEx(&lc, fused::ppo_fused_step_kernel, plan);
    if (e != cudaSuccess) {
        set_error("ppo_fused_step_kernel: launch failed: %s", cudaGetErrorString(e));
        return 2;
    }
    return 0;
}

// debug: per-phase clock64 stamps of the last step of the last launch (PPOAF_FUSED_STAMPS=1); out_host[3][kMaxPhases][4]
extern "C" int ppoaf_debug_fused_stamps(long long* out_host, int32_t* n_phase_slots) {
    if (n_phase_slots) *n_phase_slots = fused::kMaxPhases;
    if (!fused::g_stamps) return 1;
    return cudaMemcpy(out_host, fused::g_stamps, sizeof(long long) * (3 * fused::kMaxPhases * 4 + 2 * fused::kMaxPhases * 32), cudaMemcpyDeviceToHost) == cudaSuccess ? 0 : 1;
}
