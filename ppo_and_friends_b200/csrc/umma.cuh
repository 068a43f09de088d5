// tcgen05 (5th-gen tensor core) grouped GEMM for forward-only MLP launches (ppoaf_mlp_forward), fp32-accurate.
// The update never runs these tiles (their single accumulator misses its parameter tolerance, DESIGN.md §3.3), so the
// kernel carries only the forward epilogue (bias + activation) and K-major operands; the fused step kernel
// (fused_step.cu) reuses the descriptor helpers below for both operand layouts.
//
// Why tensor cores at all: the FFMA tile kernel (mlp.cuh) is bound by the per-thread
// instruction stream (~40 K warp-instructions per 32x64x256 tile); tcgen05.mma is issued by ONE
// thread and reads its operands straight from shared memory, so the threads only stage data.
// Why 3xTF32: parity with the reference needs fp32-grade products (post-epoch parameters within
// 1e-4 relative).  Every operand element x is split as hi = tf32(x), lo = tf32(x - hi) while it passes
// through registers on its way to shared memory, and D += hi*hi + hi*lo + lo*hi with fp32
// accumulation in TMEM (measured max relative error ~1e-6 on K = 64..512).
//
// Tile 128 (M) x 64 (N) per CTA, K in chunks of 32; 256 threads stage A and B (global -> registers ->
// hi/lo shared tiles, 3 stages), thread 0 issues 12 MMAs (3 terms x 4 k-steps of 8) per chunk and
// commits to an mbarrier that frees the stage; the accumulator (64 TMEM columns) is read back with
// tcgen05.ld by all 8 warps for the bias + activation epilogue.
//
// Shared-memory operand layouts (verified on hardware by scratch/umma_test.cu, scratch/umma_probe.cu):
//   K-major  operand (reduction contiguous in global; X, dZ as A;  W as B in forward):
//     SWIZZLE_128B: row r = 128 bytes (32 tf32), 16-byte chunk kq stored at (kq ^ (r & 7));
//     descriptor: start + 32 B per k-step, SBO = 1024, layout type 2.
//   MN-major operand (output dim contiguous in global; W in backward-x, dZ and X in backward-w):
//     tf32 allows ONLY SWIZZLE_128B_BASE32B: atoms of 4 k-rows x 128 B (32 outputs), 32-byte chunk c
//     stored at (c ^ (k & 3)); atoms along k at SBO = 512, groups of 32 outputs at LBO = 4096;
//     descriptor: start + 1024 B per k-step, layout type 1.
#pragma once
#include "mlp.cuh"

namespace ppoaf {
namespace umma {

constexpr int kUM = 128, kUN = 64, kUK = 32, kUStages = 3, kUThreads = 256;
constexpr int kATileFloats = kUM * kUK, kBTileFloats = kUN * kUK;
constexpr int kStageFloats = 2 * kATileFloats + 2 * kBTileFloats;       // A_hi | A_lo | B_hi | B_lo
constexpr size_t kUmmaSmemBytes = size_t(kUStages) * kStageFloats * sizeof(float) + 1024;  // + alignment slack
constexpr int kTmemCols = 64;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    return (uint64_t(layout_type) << 61) | (uint64_t(1) << 46) /* version 1 = Blackwell */ |
           (uint64_t((sbo_bytes >> 4) & 0x3FFF) << 32) | (uint64_t((lbo_bytes >> 4) & 0x3FFF) << 16) |
           uint64_t((saddr >> 4) & 0x3FFF);
}
__device__ __forceinline__ void mma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n" ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc),
        "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done = 0;
    while (!done) {
        asm volatile(
            "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
            : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    }
}
__device__ __forceinline__ float tf32_rna(float x) {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    return __uint_as_float(u);
}

// 4 consecutive floats of one row (zero beyond `n_valid`); 128-bit load when the row allows it.
__device__ __forceinline__ float4 load4(const float* __restrict__ p, int n_valid, bool vec) {
    if (n_valid <= 0) return make_float4(0.f, 0.f, 0.f, 0.f);
    if (vec && n_valid >= 4) return *reinterpret_cast<const float4*>(p);
    float4 v;
    v.x = p[0];
    v.y = n_valid > 1 ? p[1] : 0.f;
    v.z = n_valid > 2 ? p[2] : 0.f;
    v.w = n_valid > 3 ? p[3] : 0.f;
    return v;
}

// One K-major operand's per-thread staging plan: N_CH 16-byte chunks per K chunk, pointers computed once.
//   chunk (row = tid/8 + 32 i, kq = tid%8): global P[row(out0+row)*ld + k0 + 4 kq]
template <int R>
struct Stager {
    static constexpr int N_CH = R * kUK / 4 / kUThreads;   // 4 for R = 128, 2 for R = 64
    int dst[N_CH];                                         // float offset inside the tile (swizzled)
    const float* src[N_CH];                                // row base + 4 kq
    int lim[N_CH];                                         // row valid ? K : 0
    int kq4;
    bool vec;

    __device__ __forceinline__ void plan(int tid, const float* P, int ld, const int64_t* idx, int out0, int out_ext,
                                         int k_ext, bool vec_) {
        vec = vec_;
#pragma unroll
        for (int i = 0; i < N_CH; ++i) {
            const int row = tid / 8 + 32 * i, kq = tid % 8;
            dst[i] = row * 32 + ((kq ^ (row & 7)) * 4);
            const int grow = out0 + row;
            kq4 = kq * 4;
            if (grow < out_ext) {
                const int64_t r = idx ? idx[grow] : int64_t(grow);
                src[i] = P + r * ld + kq4;
                lim[i] = k_ext;
            } else {
                src[i] = P;
                lim[i] = 0;
            }
        }
    }
    __device__ __forceinline__ void load(float4 (&v)[N_CH], int k0) const {
#pragma unroll
        for (int i = 0; i < N_CH; ++i) v[i] = load4(src[i] + k0, lim[i] - (k0 + kq4), vec);
    }
    // split into hi / lo tf32 parts and store both tiles
    __device__ __forceinline__ void store(const float4 (&v)[N_CH], float* hi_tile, float* lo_tile) const {
#pragma unroll
        for (int i = 0; i < N_CH; ++i) {
            float4 h, l;
            h.x = tf32_rna(v[i].x); l.x = tf32_rna(v[i].x - h.x);
            h.y = tf32_rna(v[i].y); l.y = tf32_rna(v[i].y - h.y);
            h.z = tf32_rna(v[i].z); l.z = tf32_rna(v[i].z - h.z);
            h.w = tf32_rna(v[i].w); l.w = tf32_rna(v[i].w - h.w);
            *reinterpret_cast<float4*>(hi_tile + dst[i]) = h;
            *reinterpret_cast<float4*>(lo_tile + dst[i]) = l;
        }
    }
};

// descriptor "high" constants per operand kind; the start-address field (bits 0..13, 16-byte units) is added per use
template <bool RC>
__device__ __forceinline__ uint64_t desc_base() {
    if constexpr (RC) return make_desc(0, 0, 1024, 2);        // SWIZZLE_128B, K-major:  +32 B per k-step
    else              return make_desc(0, 4096, 512, 1);      // SWIZZLE_128B_BASE32B, MN-major: +1024 B per k-step
}
template <bool RC>
__device__ __forceinline__ uint32_t kstep_units() { return RC ? 2u : 64u; }   // 16-byte units per k-step

#ifndef PPOAF_HELPERS_ONLY
// Warp roles: warps 0..7 stage operands and run the epilogue; warp 8 (one lane) issues the MMAs.
//   full[s]  : 8 arrivals (one per staging warp, after its stores + proxy fence)  -> MMA warp may read stage s
//   free[s]  : tcgen05.commit                                                     -> stage s may be overwritten
//   acc      : tcgen05.commit after the last chunk                                 -> accumulator complete
// Y = act(X[idx] W^T + b): both operands K-major (A = X, B = W).
__device__ __forceinline__ void umma_tile(const GemmProblem& g, int tile, int64_t idx_off, float* smem, uint64_t* bars,
                                          uint32_t tmem) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = (tile / g.tiles_n) * kUM, n0 = (tile % g.tiles_n) * kUN;
    uint64_t* bar_full = bars;                    // [kUStages]
    uint64_t* bar_free = bars + kUStages;         // [kUStages]
    uint64_t* bar_acc = bars + 2 * kUStages;
    const int n_chunks = (g.K + kUK - 1) / kUK;
    PPOAF_STAMP(1);

    if (warp == kUThreads / 32) {
        // ------------------------------ MMA issuer ------------------------------
        if (lane == 0) {
            constexpr uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | (uint32_t(kUN >> 3) << 17) | (uint32_t(kUM >> 4) << 24);
            const uint64_t d0 = desc_base<true>();
            for (int c = 0; c < n_chunks; ++c) {
                const int s = c % kUStages;
                mbar_wait(&bar_full[s], uint32_t((c / kUStages) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t st = smem_u32(smem + s * kStageFloats);
                const uint64_t a_hi = d0 | uint64_t((st >> 4) & 0x3FFF);
                const uint64_t a_lo = d0 | uint64_t(((st + kATileFloats * 4) >> 4) & 0x3FFF);
                const uint64_t b_hi = d0 | uint64_t(((st + 2 * kATileFloats * 4) >> 4) & 0x3FFF);
                const uint64_t b_lo = d0 | uint64_t(((st + (2 * kATileFloats + kBTileFloats) * 4) >> 4) & 0x3FFF);
#pragma unroll
                for (uint32_t ks = 0; ks < kUK / 8; ++ks) {
                    const uint64_t o = ks * kstep_units<true>();
                    mma_tf32(tmem, a_hi + o, b_hi + o, idesc, (c > 0 || ks > 0) ? 1u : 0u);
                    mma_tf32(tmem, a_hi + o, b_lo + o, idesc, 1u);
                    mma_tf32(tmem, a_lo + o, b_hi + o, idesc, 1u);
                }
                umma_commit(&bar_free[s]);
            }
            umma_commit(bar_acc);
        }
        return;
    }

    // ------------------------------ staging warps ------------------------------
    Stager<kUM> sa;
    Stager<kUN> sb;
    sa.plan(tid, g.A, g.lda, g.idxA ? g.idxA + idx_off : nullptr, m0, g.M, g.K, (g.flavour & 2) != 0);
    sb.plan(tid, g.B, g.ldb, nullptr, n0, g.N, g.K, (g.flavour & 1) != 0);
    constexpr int NA = Stager<kUM>::N_CH, NB = Stager<kUN>::N_CH;
    float4 va[2][NA], vb[2][NB];                    // two register sets: chunk c+2 is in flight while chunk c+1 waits

    sa.load(va[0], 0);
    sb.load(vb[0], 0);
    if (n_chunks > 1) {
        sa.load(va[1], kUK);
        sb.load(vb[1], kUK);
    }
    PPOAF_STAMP(2);

    // the bias is fetched now, so its latency hides behind the main loop
    const int q = warp & 3, h = warp >> 2;
    const int m = m0 + q * 32 + lane;
    const int nb = n0 + h * 32;
    const bool vec_out = (g.ldc % 4 == 0) && (reinterpret_cast<uintptr_t>(g.C) % 16 == 0);
    // the bias keeps the alignment of the parameter buffer, which need not be 16 bytes (as in mlp.cuh's epilogue)
    const bool vec_bias = reinterpret_cast<uintptr_t>(g.bias) % 16 == 0;
    float4 bias[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int n = nb + 4 * j;
        bias[j] = n < g.N ? load4(g.bias + n, g.N - n, vec_bias) : make_float4(0.f, 0.f, 0.f, 0.f);
    }

    auto stage_chunk = [&](int c, float4 (&a_regs)[NA], float4 (&b_regs)[NB]) {
        const int s = c % kUStages;
        float* st = smem + s * kStageFloats;
        if (c >= kUStages) mbar_wait(&bar_free[s], uint32_t((c / kUStages - 1) & 1));   // MMAs of chunk c-3 have read it
        sa.store(a_regs, st, st + kATileFloats);
        sb.store(b_regs, st + 2 * kATileFloats, st + 2 * kATileFloats + kBTileFloats);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> visible to the tensor core
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(&bar_full[s])) : "memory");
        if (c + 2 < n_chunks) {
            sa.load(a_regs, (c + 2) * kUK);
            sb.load(b_regs, (c + 2) * kUK);
        }
    };
    for (int c = 0; c < n_chunks; c += 2) {
        stage_chunk(c, va[0], vb[0]);
        if (c + 1 < n_chunks) stage_chunk(c + 1, va[1], vb[1]);
    }
    PPOAF_STAMP(12);
    mbar_wait(bar_acc, 0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    PPOAF_STAMP(13);

    // ---- epilogue: warp w reads TMEM lanes 32 (w % 4) .. +31, columns 32 (w / 4) .. +31 ----
    uint32_t r[32];
    const uint32_t taddr = tmem + (uint32_t(q * 32) << 16) + uint32_t(h * 32);
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");

    if (m < g.M) {
        float* crow = g.C + int64_t(m) * g.ldc;
        const int act = g.act;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
            const int n = nb + 4 * j4;
            const float bv[4] = {bias[j4].x, bias[j4].y, bias[j4].z, bias[j4].w};
            float o[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = act_fwd_fast(__uint_as_float(r[4 * j4 + j]) + bv[j], act);
            if (vec_out && n + 3 < g.N) {
                *reinterpret_cast<float4*>(crow + n) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (n + j < g.N) crow[n + j] = o[j];
            }
        }
    }
    PPOAF_STAMP(14);
}

__global__ void __launch_bounds__(kUThreads + 32) umma_grouped_gemm_kernel(const GroupedGemmArgs args) {
    extern __shared__ uint8_t smem_raw[];
    PPOAF_STAMP(0);
    __shared__ __align__(8) uint64_t s_bars[2 * kUStages + 1];
    __shared__ uint32_t s_tmem;
    float* smem = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    const int tid = threadIdx.x, warp = tid >> 5;

    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&s_tmem)), "r"(kTmemCols));
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
    }
    if (tid == 32) {
#pragma unroll
        for (int i = 0; i < kUStages; ++i) {
            mbar_init(&s_bars[i], kUThreads / 32);            // full: one arrival per staging warp
            mbar_init(&s_bars[kUStages + i], 1);              // free: tcgen05.commit
        }
        mbar_init(&s_bars[2 * kUStages], 1);                  // accumulator complete
        asm volatile("fence.mbarrier_init.release.cluster;");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = s_tmem;

    int p = 0;
#pragma unroll
    for (int i = 1; i < kMaxGroup; ++i)
        if (i < args.n_problems && int(blockIdx.x) >= args.p[i].tile_begin) p = i;
    const GemmProblem& g = args.p[p];
    const int tile = int(blockIdx.x) - g.tile_begin;
    pdl_wait();
    pdl_trigger();
    const int64_t idx_off = args.cursor ? int64_t(*args.cursor) * args.cursor_stride : 0;
    umma_tile(g, tile, idx_off, smem, s_bars, tmem);

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"(kTmemCols));
}

#endif  // PPOAF_HELPERS_ONLY

}  // namespace umma
}  // namespace ppoaf
