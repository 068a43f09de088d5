// Segment table -> flat map, and GAE + reward-to-go as one segmented reverse scan with
// decoupled look-back (single pass over HBM: 17 B/timestep + 9 B/segment).
//
// Reference arithmetic restated (utils/episode_info.py:254-260, 289-293, 410-417, 450-461):
//   V^_t = f32(V_t), V^_L = f32(v_boot);  delta_t = r_t + f32(gamma_f32 * V^_{t+1}) - V^_t  (f64 sum)
//   A_t  = delta_t + (gamma*lambda) A_{t+1},  A_L = 0                                        (f64)
//   RTG_t = f32(r_t) + gamma RTG_{t+1},  RTG_L = f32(clip(r_boot))                             (f64)
// Each element is the affine map x -> a + b x (b = 0 at a segment's last element, where the
// seeds enter through a); maps compose associatively, so the reverse scan parallelises.
// A map that contains a segment end carries the bit `e` and is the constant a: the value from the right is DROPPED
// there, not multiplied by zero, so a NaN or Inf stays inside its own segment (IEEE 0 * NaN = 0 * Inf = NaN) as it
// does in the per-episode reference.  b == 0 is not such a test: it also holds inside a segment when gamma*lambda is 0
// or gamma*lambda^k underflows, where the reference does propagate a NaN.
#include "common.cuh"

namespace ppoaf {

// ------------------------------------------------------------------------------------------------
__global__ void build_flat_map_kernel(const int32_t* __restrict__ seg_col, const int32_t* __restrict__ seg_t0,
                                      const int32_t* __restrict__ seg_len, const int64_t* __restrict__ seg_off,
                                      const uint8_t* __restrict__ seg_terminal, int32_t n_seg, int32_t n_cols,
                                      int32_t* __restrict__ src_row, uint8_t* __restrict__ seg_flag) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = (int64_t(gridDim.x) * blockDim.x) >> 5;
    for (int64_t s = warp; s < n_seg; s += nwarps) {
        const int32_t col = seg_col[s], t0 = seg_t0[s], len = seg_len[s];
        const int64_t off = seg_off[s];
        const uint8_t endflag = uint8_t(1u | (seg_terminal[s] ? 2u : 0u));
        for (int32_t k = lane; k < len; k += 32) {
            src_row[off + k] = (t0 + k) * n_cols + col;
            seg_flag[off + k] = (k == len - 1) ? endflag : uint8_t(0);
        }
    }
}

// ------------------------------------------------------------------------------------------------
struct Affine2 {  // advantage map (aA, bA) and reward-to-go map (aR, bR); e: the range contains a segment end
    double aA, bA, aR, bR;
    int e;
};
// result(x) = l(r(x)): l is the element/range on the LEFT (lower index), applied after r.
__device__ __forceinline__ Affine2 compose(const Affine2& l, const Affine2& r) {
    Affine2 o;
    o.aA = l.e ? l.aA : fma(l.bA, r.aA, l.aA);
    o.bA = l.bA * r.bA;
    o.aR = l.e ? l.aR : fma(l.bR, r.aR, l.aR);
    o.bR = l.bR * r.bR;
    o.e = l.e | r.e;
    return o;
}
// m(x) for a value x entering from the right of the range m
__device__ __forceinline__ double apply_adv(const Affine2& m, double x) { return m.e ? m.aA : fma(m.bA, x, m.aA); }
__device__ __forceinline__ double apply_rtg(const Affine2& m, double x) { return m.e ? m.aR : fma(m.bR, x, m.aR); }
__device__ __forceinline__ Affine2 shfl_down_affine(const Affine2& v, int d) {
    Affine2 o;
    o.aA = __shfl_down_sync(kFull, v.aA, d);
    o.bA = __shfl_down_sync(kFull, v.bA, d);
    o.aR = __shfl_down_sync(kFull, v.aR, d);
    o.bR = __shfl_down_sync(kFull, v.bR, d);
    o.e = __shfl_down_sync(kFull, v.e, d);
    return o;
}

struct alignas(64) TileDesc {
    double aA, bA, aR, bR;  // tile aggregate map
    double vA, vR;          // A and RTG at the tile's first (lowest) element
    int status;             // 0 = empty, 1 = aggregate ready, 2 = value ready
    int e;                  // the tile contains a segment end
};

__device__ __forceinline__ int ld_acquire(const int* p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release(int* p, int v) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

constexpr int kScanThreads = 128;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;  // 1024 timesteps per CTA


// Staged inputs of one tile (double-buffered with cp.async: the next tile of this CTA travels while the current one is
// scanned): rewards, values (+ the one-element halo V_{t+1} of the tile's last element) and the segment-end flags.
struct ScanStage {
    float r[kScanTile];
    float v[kScanTile + 4];
    uint8_t f[kScanTile];
};

__device__ __forceinline__ void scan_cp16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(smem_dst))), "l"(gsrc)
                 : "memory");
}
__device__ __forceinline__ void scan_cp8(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(smem_dst))), "l"(gsrc)
                 : "memory");
}
__device__ __forceinline__ void scan_cp4(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(static_cast<unsigned>(__cvta_generic_to_shared(smem_dst))), "l"(gsrc)
                 : "memory");
}

// first segment that intersects a tile: last s with seg_off[s] <= lo.  A 32-ary search by one warp: every step probes 32
// positions at once, so 115 K segments take 4 dependent loads instead of 17.
__device__ __forceinline__ int first_segment_of(const int64_t* __restrict__ seg_off, int n_seg, int64_t lo, int lane) {
    int a = 0, b = n_seg;  // invariant: seg_off[a] <= lo < seg_off[b]  (b == n_seg is a virtual +inf)
    while (b - a > 1) {
        const int step = (b - a + 31) / 32;
        const int probe = a + (lane + 1) * step;
        const bool le = probe < b && seg_off[probe] <= lo;
        const unsigned m = __ballot_sync(kFull, le);            // monotone: the first k lanes are true
        const int k = __popc(m);
        const int na = a + k * step;
        b = min(b, na + step);
        a = na;
    }
    return a;
}

// PERSISTENT: the grid holds at most as many CTAs as can be resident at once (host: occupancy x SMs) and CTA b scans
// tiles T-1-b, T-1-b-G, ... (highest first: the scan runs right to left).  A tile only ever waits on HIGHER tiles, which
// belong to CTAs that are resident or can become resident without anyone's help, and every CTA takes its own tiles in
// descending order - so the look-back cannot deadlock whatever order the hardware dispatches thread blocks in (round 1
// relied on blockIdx-order dispatch).  No atomic ticket is needed: the assignment is static.
__global__ void __launch_bounds__(kScanThreads, 8)
segscan_kernel(const float* __restrict__ rewards, const float* __restrict__ values,
               const uint8_t* __restrict__ seg_flag, const int64_t* __restrict__ seg_off,
               const float* __restrict__ v_boot, const float* __restrict__ r_boot, int32_t n_seg, int64_t n,
               double gamma, double gamma_lambda, float gamma_f, int use_gae, float* __restrict__ adv_out,
               float* __restrict__ rtg_out, TileDesc* __restrict__ desc, int n_tiles) {
    __shared__ __align__(16) ScanStage s_in[2];
    __shared__ int s_warp_ends[kScanThreads / 32];
    __shared__ Affine2 s_warp_agg[kScanThreads / 32];
    __shared__ int s_first_seg[2];
    __shared__ double s_carry[2];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int G = int(gridDim.x);
    const int i0 = tid * kScanItems;

    auto stage_tile = [&](int t, ScanStage& st) {
        const int64_t lo = int64_t(t) * kScanTile;
        const int64_t hi = min(lo + int64_t(kScanTile), n);
        const int cnt = int(hi - lo);
        if (cnt == kScanTile) {                     // every tile but (possibly) the last: 16-byte async copies
            scan_cp16(&st.r[4 * tid], rewards + lo + 4 * tid);
            scan_cp16(&st.r[4 * (tid + kScanThreads)], rewards + lo + 4 * (tid + kScanThreads));
            scan_cp16(&st.v[4 * tid], values + lo + 4 * tid);
            scan_cp16(&st.v[4 * (tid + kScanThreads)], values + lo + 4 * (tid + kScanThreads));
            scan_cp8(&st.f[8 * tid], seg_flag + lo + 8 * tid);          // flags are only 8-byte aligned
            if (tid == kScanThreads - 1) {
                if (hi < n) scan_cp4(&st.v[kScanTile], values + hi);
                else st.v[kScanTile] = 0.f;
            }
        } else {                                    // ragged last tile: guarded loads, padding = inert one-element segments
            for (int k = tid; k < kScanTile; k += kScanThreads) {
                const bool in = k < cnt;
                st.r[k] = in ? rewards[lo + k] : 0.f;
                st.v[k] = in ? values[lo + k] : 0.f;
                st.f[k] = in ? seg_flag[lo + k] : uint8_t(1);
            }                                       // (a ragged tile is the last one: its halo st.v[cnt] is the padding zero)
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };

    int tile = n_tiles - 1 - int(blockIdx.x);
    if (tile < 0) return;
    stage_tile(tile, s_in[0]);
    if (warp == 1) {
        const int a = first_segment_of(seg_off, n_seg, int64_t(tile) * kScanTile, lane);
        if (lane == 0) s_first_seg[0] = a;
    }

#pragma unroll 1
    for (int it = 0; tile >= 0; ++it, tile -= G) {
        const int cur = it & 1;
        const int next_tile = tile - G;
        if (next_tile >= 0) stage_tile(next_tile, s_in[cur ^ 1]);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");       // the current tile has landed (the next may be in flight)
        __syncthreads();
        const ScanStage& st = s_in[cur];
        const int64_t lo = int64_t(tile) * kScanTile;
        const int64_t hi = min(lo + int64_t(kScanTile), n);
        const int cnt = int(hi - lo);

        float r[kScanItems], v[kScanItems];
        uint8_t f[kScanItems];
        {
            const float4 ra = *reinterpret_cast<const float4*>(&st.r[i0]), rb = *reinterpret_cast<const float4*>(&st.r[i0 + 4]);
            const float4 va = *reinterpret_cast<const float4*>(&st.v[i0]), vb = *reinterpret_cast<const float4*>(&st.v[i0 + 4]);
            r[0] = ra.x; r[1] = ra.y; r[2] = ra.z; r[3] = ra.w; r[4] = rb.x; r[5] = rb.y; r[6] = rb.z; r[7] = rb.w;
            v[0] = va.x; v[1] = va.y; v[2] = va.z; v[3] = va.w; v[4] = vb.x; v[5] = vb.y; v[6] = vb.z; v[7] = vb.w;
            const uint2 fw = *reinterpret_cast<const uint2*>(&st.f[i0]);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                f[k] = uint8_t(fw.x >> (8 * k));
                f[4 + k] = uint8_t(fw.y >> (8 * k));
            }
        }

        // ---- ordinal of every segment end inside the tile -> which seeds it takes ----
        int my_ends = 0;
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) my_ends += (f[k] & 1) && (i0 + k < cnt);
        int ends_incl = my_ends;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFull, ends_incl, o);
            if (lane >= o) ends_incl += t;
        }
        if (lane == 31) s_warp_ends[warp] = ends_incl;
        __syncthreads();
        int ends_before = ends_incl - my_ends;
        for (int w = 0; w < warp; ++w) ends_before += s_warp_ends[w];
        int seg = s_first_seg[cur] + ends_before;

        // ---- per-element maps, composed right-to-left inside the thread ----
        double a_adv[kScanItems], a_rtg[kScanItems];
        uint32_t endmask = 0;
#pragma unroll
        for (int k = 0; k < kScanItems; ++k) {
            const bool in = i0 + k < cnt;
            const bool end = (f[k] & 1) != 0;
            float vnext = st.v[min(i0 + k + 1, kScanTile)];
            if (i0 + k + 1 == cnt) vnext = st.v[cnt];               // ragged tile: the halo sits right after the last element
            double rt = double(r[k]);
            double aR = rt;
            if (end) {
                if (in) {
                    vnext = v_boot[seg];
                    aR = fma(gamma, double(r_boot[seg]), rt);
                    ++seg;
                } else {
                    vnext = 0.f;
                }
                endmask |= 1u << k;
            }
            a_adv[k] = rt + double(__fmul_rn(gamma_f, vnext)) - double(v[k]);
            a_rtg[k] = aR;
        }
        Affine2 agg;  // identity
        agg.aA = 0.0; agg.bA = 1.0; agg.aR = 0.0; agg.bR = 1.0; agg.e = 0;
#pragma unroll
        for (int k = kScanItems - 1; k >= 0; --k) {
            Affine2 e;
            const bool end = (endmask >> k) & 1u;
            e.aA = a_adv[k]; e.bA = end ? 0.0 : gamma_lambda;
            e.aR = a_rtg[k]; e.bR = end ? 0.0 : gamma;
            e.e = end;
            agg = compose(e, agg);
        }

        // ---- reverse scan across the warp: suffix[t] = agg[t] o agg[t+1] o ... o agg[31] ----
        Affine2 suffix = agg;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const Affine2 right = shfl_down_affine(suffix, o);
            if (lane + o < 32) suffix = compose(suffix, right);
        }
        if (lane == 0) s_warp_agg[warp] = suffix;
        __syncthreads();
        Affine2 right_in_tile;
        right_in_tile.aA = 0.0; right_in_tile.bA = 1.0; right_in_tile.aR = 0.0; right_in_tile.bR = 1.0; right_in_tile.e = 0;
        {
            const Affine2 lane_right = shfl_down_affine(suffix, 1);
            if (lane < 31) right_in_tile = lane_right;
            for (int w = warp + 1; w < kScanThreads / 32; ++w) right_in_tile = compose(right_in_tile, s_warp_agg[w]);
        }

        // ---- decoupled look-back over the tiles to the right (thread 0), while warp 1 finds the first segment of this
        // CTA's NEXT tile ----
        if (warp == 1 && next_tile >= 0) {
            const int a = first_segment_of(seg_off, n_seg, int64_t(next_tile) * kScanTile, lane);
            if (lane == 0) s_first_seg[cur ^ 1] = a;
        }
        if (tid == 0) {
            Affine2 tile_agg = s_warp_agg[0];
            for (int w = 1; w < kScanThreads / 32; ++w) tile_agg = compose(tile_agg, s_warp_agg[w]);
            TileDesc* d = desc + tile;
            const bool closed = tile_agg.e || tile == n_tiles - 1;
            d->aA = tile_agg.aA; d->bA = tile_agg.bA; d->aR = tile_agg.aR; d->bR = tile_agg.bR; d->e = tile_agg.e;
            if (closed) {  // carry-in is dropped at a segment end (or is zero past the end): value known at once
                d->vA = tile_agg.aA; d->vR = tile_agg.aR;
                __threadfence();
                st_release(&d->status, 2);
            } else {
                __threadfence();
                st_release(&d->status, 1);
            }
            double cA = 0.0, cR = 0.0;  // carry entering the tile from the right
            if (tile != n_tiles - 1) {
                Affine2 acc;  // composition of the tiles inspected so far
                acc.aA = 0.0; acc.bA = 1.0; acc.aR = 0.0; acc.bR = 1.0; acc.e = 0;
                int k = tile + 1;
                while (true) {
                    if (k == n_tiles) { cA = acc.aA; cR = acc.aR; break; }
                    const TileDesc* p = desc + k;
                    int stt;
                    do { stt = ld_acquire(&p->status); } while (stt == 0);
                    if (stt == 2) {  // acc has no segment end here: the loop leaves as soon as it gains one
                        cA = fma(acc.bA, __ldcg(&p->vA), acc.aA);
                        cR = fma(acc.bR, __ldcg(&p->vR), acc.aR);
                        break;
                    }
                    Affine2 t;
                    t.aA = __ldcg(&p->aA); t.bA = __ldcg(&p->bA); t.aR = __ldcg(&p->aR); t.bR = __ldcg(&p->bR);
                    t.e = __ldcg(&p->e);
                    acc = compose(acc, t);
                    if (acc.e) { cA = acc.aA; cR = acc.aR; break; }
                    ++k;
                }
                if (!closed) {  // (no segment end in the tile)
                    d->vA = fma(tile_agg.bA, cA, tile_agg.aA);
                    d->vR = fma(tile_agg.bR, cR, tile_agg.aR);
                    __threadfence();
                    st_release(&d->status, 2);
                }
            }
            s_carry[0] = cA; s_carry[1] = cR;
        }
        __syncthreads();

        // ---- apply: values right of this thread, then walk the thread's items right to left ----
        double xA = apply_adv(right_in_tile, s_carry[0]);
        double xR = apply_rtg(right_in_tile, s_carry[1]);
        float oa[kScanItems], og[kScanItems];
#pragma unroll
        for (int k = kScanItems - 1; k >= 0; --k) {
            const bool end = (endmask >> k) & 1u;
            xA = end ? a_adv[k] : fma(gamma_lambda, xA, a_adv[k]);
            xR = end ? a_rtg[k] : fma(gamma, xR, a_rtg[k]);
            og[k] = float(xR);
            oa[k] = use_gae ? float(xA) : float(xR - double(v[k]));
        }
        if (cnt == kScanTile) {
            float4* a4 = reinterpret_cast<float4*>(adv_out + lo + i0);
            float4* g4 = reinterpret_cast<float4*>(rtg_out + lo + i0);
            stg_stream_f4(a4, make_float4(oa[0], oa[1], oa[2], oa[3]));
            stg_stream_f4(a4 + 1, make_float4(oa[4], oa[5], oa[6], oa[7]));
            stg_stream_f4(g4, make_float4(og[0], og[1], og[2], og[3]));
            stg_stream_f4(g4 + 1, make_float4(og[4], og[5], og[6], og[7]));
        } else {
#pragma unroll
            for (int k = 0; k < kScanItems; ++k)
                if (i0 + k < cnt) {
                    adv_out[lo + i0 + k] = oa[k];
                    rtg_out[lo + i0 + k] = og[k];
                }
        }
        // the shared arrays (stage `cur`, warp aggregates, carry) are rewritten by the next iteration only after its first
        // __syncthreads, which every thread reaches after finishing this one
    }
    asm volatile("cp.async.wait_group 0;" ::: "memory");
}

}  // namespace ppoaf


using namespace ppoaf;

extern "C" int ppoaf_build_flat_map(const int32_t* seg_col, const int32_t* seg_t0, const int32_t* seg_len,
                                    const int64_t* seg_off, const uint8_t* seg_terminal, int32_t n_seg,
                                    int32_t n_cols, int64_t n_flat, int32_t* src_row, uint8_t* seg_flag,
                                    void* stream) {
    PPOAF_CHECK_ARG(n_seg >= 0 && n_cols > 0 && n_flat >= 0, "ppoaf_build_flat_map: bad sizes");
    PPOAF_CHECK_ARG(n_flat < (int64_t(1) << 31), "ppoaf_build_flat_map: ring rows are int32: n_flat must stay below 2^31");
    if (n_seg == 0) return 0;
    const int threads = 256;
    int64_t blocks = ceil_div64(int64_t(n_seg) * 32, threads);
    const int64_t cap = int64_t(sm_count()) * 16;
    if (blocks > cap) blocks = cap;
    build_flat_map_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(
        seg_col, seg_t0, seg_len, seg_off, seg_terminal, n_seg, n_cols, src_row, seg_flag);
    PPOAF_CHECK_LAUNCH("ppoaf_build_flat_map");
    return 0;
}

extern "C" size_t ppoaf_segscan_workspace_bytes(int64_t n_flat) {
    const int64_t tiles = ceil_div64(n_flat > 0 ? n_flat : 1, kScanTile);
    return size_t(tiles) * sizeof(TileDesc) + 64;
}

extern "C" int ppoaf_gae_rtg_segscan(const float* rewards, const float* values, const uint8_t* seg_flag,
                                     const int64_t* seg_off, const float* v_boot, const float* r_boot,
                                     int32_t n_seg, int64_t n_flat, double gamma, double lambd, int use_gae,
                                     float* adv_out, float* rtg_out, void* workspace, size_t workspace_bytes,
                                     void* stream) {
    PPOAF_CHECK_ARG(n_flat >= 0 && n_seg >= 0, "ppoaf_gae_rtg_segscan: bad sizes");
    if (n_flat == 0) return 0;
    PPOAF_CHECK_ARG(n_seg > 0, "ppoaf_gae_rtg_segscan: n_flat > 0 needs at least one segment");
    PPOAF_CHECK_ARG(workspace_bytes >= ppoaf_segscan_workspace_bytes(n_flat),
                    "ppoaf_gae_rtg_segscan: workspace too small");
    PPOAF_CHECK_ARG((reinterpret_cast<uintptr_t>(rewards) | reinterpret_cast<uintptr_t>(values) |
                     reinterpret_cast<uintptr_t>(adv_out) | reinterpret_cast<uintptr_t>(rtg_out)) % 16 == 0 &&
                        reinterpret_cast<uintptr_t>(seg_flag) % 8 == 0 &&
                        reinterpret_cast<uintptr_t>(workspace) % 64 == 0,
                    "ppoaf_gae_rtg_segscan: buffers must be 16-byte aligned (flags 8, workspace 64)");
    const int n_tiles = int(ceil_div64(n_flat, kScanTile));
    cudaStream_t s = (cudaStream_t)stream;
    // descriptors + ticket are reset every launch (a memset node when captured in a graph)
    cudaError_t e = cudaMemsetAsync(workspace, 0, ppoaf_segscan_workspace_bytes(n_flat), s);
    PPOAF_CHECK_ARG(e == cudaSuccess, "ppoaf_gae_rtg_segscan: memset failed: %s", cudaGetErrorString(e));
    TileDesc* desc = reinterpret_cast<TileDesc*>(workspace);
    // persistent grid: no more CTAs than can be resident at once (see the kernel's forward-progress argument)
    static int resident = 0;
    if (resident == 0) {
        int per_sm = 0;
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, segscan_kernel, kScanThreads, 0) != cudaSuccess || per_sm < 1) {
            (void)cudaGetLastError();
            per_sm = 1;
        }
        resident = per_sm * sm_count();
    }
    const int grid = n_tiles < resident ? n_tiles : resident;
    segscan_kernel<<<grid, kScanThreads, 0, s>>>(rewards, values, seg_flag, seg_off, v_boot, r_boot, n_seg, n_flat, gamma,
                                                 gamma * lambd, float(gamma), use_gae, adv_out, rtg_out, desc, n_tiles);
    PPOAF_CHECK_LAUNCH("ppoaf_gae_rtg_segscan");
    return 0;
}
