// composite_fwd / composite_bwd: per-tile front-to-back alpha blending and its backward.
//
// Replaces upstream's renderCUDA forward/backward (SURVEY.md 2.4 K6/K7, App. A.6/A.7; restated
// in oracle/splat_ref.py::composite).  B200 design:
//   * persistent CTAs pull work from a queue ordered longest-list-first.  FORWARD: a CTA
//     (8 warps x (8x4)-pixel blocks) takes a whole 16x16 tile and shares every gathered chunk;
//     BACKWARD: every warp is an independent worker on one 8x4 block (lists are truncated at the
//     block's own last contributor, so there is no long scan to share and no CTA barrier at all);
//   * a tile's list is its contiguous range of the depth-sorted key array; per chunk of 256
//     entries every thread reads ONE key (coalesced 8-B loads, prefetched two chunks ahead in a
//     register) and copies that Gaussian's 48-byte record from the L2-resident per-Gaussian array
//     straight into a double-buffered shared-memory ring with three 16-byte cp.async (LDGSTS):
//     no register staging, the copies for chunk c+1 fly while chunk c is being blended, and
//     - because saturated tiles stop early - records past the stopping point are never fetched;
//   * each warp tests 32 records at a time (one per lane) against its own 8x4 pixel block
//     (conservative extent test, never changes which pixels blend) and only evaluates the
//     survivors, in list order, reading them back with broadcast LDS.128;
//   * forward: warp/CTA early-out when every pixel is saturated (T < 1e-4 would follow);
//   * backward: per-(warp, Gaussian) partial gradients are reduced with a halving shuffle
//     butterfly (12 SHFL for 10 values) and committed with ONE coalesced RED instruction.
#include "common.cuh"
#include <cuda_fp16.h>

namespace {

// BACKWARD work item = one warp's 8x4 pixel block of one non-empty tile (8 items per tile, queue
// ordered longest list first).  Every warp is an independent worker with a private ring of kSlots
// sub-chunks (32 records = one per lane): the backward kernel contains no CTA-wide barrier.
constexpr int kWarps = 8;      // warps per CTA (in the backward kernel just a container)
constexpr int kSlots = 3;      // sub-chunks in the ring per warp (kSlots-1 being gathered + 1 being blended)
constexpr int kMinCtas = 4;    // backward CTAs per SM
struct __align__(128) SmemRing {
    GsrRec rec[kWarps][kSlots][32];   // 1.5 KB per slot and warp
};

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }

// copy geom[idx(key)] into rec (3 x 16 B)
__device__ __forceinline__ void gather_record(GsrRec* rec, const GsrRec* __restrict__ geom,
                                              unsigned long long key) {
    const char* src = reinterpret_cast<const char*>(geom + (uint32_t)key);
    char* dst = reinterpret_cast<char*>(rec);
    cp_async16(dst, src);
    cp_async16(dst + 16, src + 16);
    cp_async16(dst + 32, src + 32);
}

// Forward epilogue: a block that blended at least one entry becomes a work item of the backward, filed under
// the size class of its consumed list length (see GSR_BWD_CLASSES).  `n` is warp-uniform; call from lane 0.
__device__ __forceinline__ void bwd_item_append(uint32_t* fill, uint32_t* items, int ntiles, uint32_t tile,
                                                int blk, uint32_t n) {
    if (items == nullptr || n == 0u) return;
    const int k = gsr_bwd_class(n);
    const uint32_t slot = atomicAdd(fill + k, 1u);
    items[(size_t)k * ntiles * 8 + slot] = tile * 8u + (uint32_t)blk;
}

// The blending test, shared verbatim by forward and backward so both take identical decisions.
struct PairEval {
    float dx, dy, G, alpha;
    bool valid;
};
__device__ __forceinline__ PairEval eval_pair(float px, float py, float A, float B, float C,
                                              float opacity, float X, float Y) {
    PairEval e;
    const float2 d2 = __fadd2_rn(make_float2(px, py), make_float2(-X, -Y));     // one FADD2
    e.dx = d2.x;
    e.dy = d2.y;
#ifdef GSR_EXACT_EXP
    // oracle order (splat_ref.py::composite): power = -0.5*(A*dx*dx + C*dy*dy) - B*dx*dy, raw conic
    const float qs = __fadd_rn(__fmul_rn(__fmul_rn(A, e.dx), e.dx), __fmul_rn(__fmul_rn(C, e.dy), e.dy));
    const float p2 = __fsub_rn(__fmul_rn(-0.5f, qs), __fmul_rn(__fmul_rn(B, e.dx), e.dy));
    e.G = expf(fminf(p2, 0.0f));
#else
    const float u = __fmaf_rn(A, e.dx, __fmul_rn(B, e.dy));
    const float p2 = __fmaf_rn(__fmul_rn(C, e.dy), e.dy, __fmul_rn(u, e.dx));
    e.G = ex2_approx(p2);
#endif
    e.alpha = fminf(GSR_ALPHA_MAX, __fmul_rn(opacity, e.G));
    e.valid = (p2 <= 0.0f) && (e.alpha >= GSR_ALPHA_MIN);
    return e;
}

__device__ __forceinline__ bool cull_pass(float px, float py, uint32_t ext, float X0, float Y0) {
    // block covers pixel centres [X0, X0+7] x [Y0, Y0+3]
    const __half2 eh = *reinterpret_cast<const __half2*>(&ext);
    const float2 e = __half22float2(eh);
    const float ddx = fmaxf(fmaxf(X0 - px, px - (X0 + 7.0f)), 0.0f);
    const float ddy = fmaxf(fmaxf(Y0 - py, py - (Y0 + 3.0f)), 0.0f);
    return (ddx <= e.x) && (ddy <= e.y);
}

// slots of the optional diagnostic counters (b200gsr_debug_counters)
enum { GSR_STAT_BWD_EVAL = 0, GSR_STAT_BWD_CONTRIB = 1, GSR_STAT_BWD_LANES = 2, GSR_STAT_BWD_HIST = 3,   // 3..8
       GSR_STAT_FWD_EVAL = 10, GSR_STAT_FWD_LANES = 11,
       // load balance of the persistent kernels (globaltimer ns): sum of worker busy time, last exit,
       // ~(first entry) [so that atomicMax on a zeroed word yields the minimum], workers, largest item
       GSR_STAT_FWD_BUSY = 16, GSR_STAT_FWD_END = 17, GSR_STAT_FWD_NBEGIN = 18, GSR_STAT_FWD_WORKERS = 19,
       GSR_STAT_FWD_MAX_ITEM = 20,
       GSR_STAT_BWD_BUSY = 21, GSR_STAT_BWD_END = 22, GSR_STAT_BWD_NBEGIN = 23, GSR_STAT_BWD_WORKERS = 24,
       GSR_STAT_BWD_MAX_ITEM = 25, GSR_STAT_BWD_MAX_ITEM_NS = 26, GSR_STAT_WORDS = 32 };
__device__ __forceinline__ unsigned long long gsr_now_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

// =============================================================================================
// Forward
// =============================================================================================
// Forward keeps the tile as the unit of work: blocks that never saturate (silhouettes, thin
// regions) must scan the whole list, and sharing each gathered 256-entry chunk between the 8
// warps of the tile makes that scan cheap (measured: 0.145 ms vs 0.170 ms for independent warps).
constexpr int kChunk = 256;   // list entries per pipeline stage (kChunk/256 per thread)
struct __align__(128) SmemCta {
    GsrRec rec[2][kChunk];   // 2 x 12 KB at kChunk = 256
    uint32_t work;           // broadcast slot for the tile queue
};

// One CTA of 256/PPL threads per tile; each warp renders an 8x(4*PPL)-pixel block.  Only PPL = 1 (one pixel
// per lane) is instantiated: 2 pixels per lane lost in round 1.
template <bool SCORE, int PPL, bool STATS>
__global__ void __launch_bounds__(256 / PPL)
composite_fwd_kernel(int H, int W, int gx, int gy_view, int Hs, int ntiles, const uint32_t* __restrict__ header,
                     const uint32_t* __restrict__ work_order,
                     const uint32_t* __restrict__ tile_start,
                     const unsigned long long* __restrict__ keys, const GsrRec* __restrict__ geom,
                     const float* __restrict__ bg, uint32_t* __restrict__ queue,
                     float* __restrict__ out_color, float* __restrict__ out_depth_alpha,
                     uint32_t* __restrict__ n_contrib, float* __restrict__ score,
                     unsigned long long* __restrict__ stats, uint32_t* bwd_fill, uint32_t* bwd_items) {
    constexpr int kThreads = 256 / PPL;
    unsigned int st_eval = 0, st_lanes = 0;
    unsigned long long st_t0 = 0, st_item_t0 = 0, st_max_item_ns = 0;
    if (STATS) st_t0 = gsr_now_ns();
    constexpr int kPer = kChunk / kThreads;   // list entries gathered per thread per chunk
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemCta& sm = *reinterpret_cast<SmemCta*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const uint32_t max_pairs = header[GSR_H_MAX_PAIRS];

    for (;;) {
        // one shared counter over ALL tiles (empty ones included, they come last): measured faster
        // here than the split queue + static empty tiles (0.141 vs 0.157 ms)
        if (STATS) {
            const unsigned long long t = gsr_now_ns();
            if (st_item_t0 && t - st_item_t0 > st_max_item_ns) st_max_item_ns = t - st_item_t0;
            st_item_t0 = t;
        }
        if (tid == 0) sm.work = atomicAdd(queue, 1u);
        __syncthreads();
        const uint32_t w = sm.work;
        __syncthreads();   // everyone has read the slot before thread 0 may overwrite it
        if (w >= (uint32_t)ntiles) break;
        const uint32_t tile = work_order[w];
        const int blk = wid;      // 8x(4*PPL)-pixel block of the tile this warp renders
        uint32_t beg = tile_start[tile], end = tile_start[tile + 1];
        if (end > max_pairs) end = max_pairs;
        if (beg > end) beg = end;
        const int n = (int)(end - beg);
        const int nchunks = (n + kChunk - 1) / kChunk;
        const unsigned long long* tk = keys + beg;
        const int tys = tile / gx, txi = tile - tys * gx;
        // multi-view: tile row tys of the stacked image = row tyi of view `view`; everything is evaluated in
        // view-local pixel coordinates (bit-identical to a single-view render), only addressing is stacked
        const int view = tys / gy_view, tyi = tys - view * gy_view;
        const int row0 = view * gy_view * GSR_TILE;
        const float* bgv = bg + 3 * view;
        const float bg0 = __ldg(bgv), bg1 = __ldg(bgv + 1), bg2 = __ldg(bgv + 2);
        const int X0i = txi * GSR_TILE + (blk & 1) * 8, Y0i = tyi * GSR_TILE + (blk >> 1) * (4 * PPL);
        const int Xi = X0i + (lane & 7), Yi = Y0i + (lane >> 3);
        const float X0 = (float)X0i, Y0 = (float)Y0i, X = (float)Xi;
        bool inside[PPL], done[PPL];
        float Y[PPL], T[PPL];
        float2 C01[PPL], C2D[PPL];         // (r, g) and (b, depth) accumulators: two FFMA2 per blend
        uint32_t last[PPL];
        bool all_done = true;
#pragma unroll
        for (int q = 0; q < PPL; ++q) {
            inside[q] = Xi < W && (Yi + 4 * q) < H;
            done[q] = !inside[q];
            all_done = all_done && done[q];
            Y[q] = (float)(Yi + 4 * q);
            T[q] = 1.0f; C01[q] = make_float2(0.f, 0.f); C2D[q] = make_float2(0.f, 0.f); last[q] = 0;
        }

        // prologue: gather chunk 0, prefetch the keys of chunk 1
        unsigned long long knext[kPer];
#pragma unroll
        for (int u = 0; u < kPer; ++u) {
            const int e = u * kThreads + tid;
            if (e < n) gather_record(&sm.rec[0][e], geom, __ldg(tk + e));
            knext[u] = (kChunk + e < n) ? __ldg(tk + kChunk + e) : 0ull;
        }
        cp_async_commit();

        for (int c = 0; c < nchunks; ++c) {
            cp_async_wait<0>();   // my copies for chunk c have landed
            // barrier: everyone's copies for chunk c are visible, everyone is done with chunk c-1;
            // it doubles as the CTA-wide early-out vote
            const int ndone = __syncthreads_count(all_done);
            if (ndone == kThreads) break;
            // issue the gathers for chunk c+1 (they fly while chunk c is blended), then fetch the
            // keys of chunk c+2
#pragma unroll
            for (int u = 0; u < kPer; ++u) {
                const int e = u * kThreads + tid;
                if ((c + 1) * kChunk + e < n) gather_record(&sm.rec[(c + 1) & 1][e], geom, knext[u]);
                knext[u] = ((c + 2) * kChunk + e < n) ? __ldg(tk + (c + 2) * kChunk + e) : 0ull;
            }
            cp_async_commit();

            const GsrRec* st = sm.rec[c & 1];
            const int cnt = min(kChunk, n - c * kChunk);
            if (__all_sync(0xffffffffu, all_done)) continue;   // this warp is saturated
            for (int sub = 0; sub * 32 < cnt; ++sub) {
                const int r = sub * 32 + lane;
                bool pass = false;
                if (r < cnt) {
                    const float4 q0 = *reinterpret_cast<const float4*>(&st[r]);
                    pass = cull_pass(q0.x, q0.y, __float_as_uint(q0.z), X0, Y0);
                }
                uint32_t mask = __ballot_sync(0xffffffffu, pass);
                const float4* sp = reinterpret_cast<const float4*>(&st[sub * 32]);
                const uint32_t pos0 = (uint32_t)(c * kChunk + sub * 32 + 1);
                // One list entry applied to this lane's pixel(s): the T / colour recurrences are the only
                // dependences between consecutive entries.
                auto blend = [&](const float4& q1, const float4& q2, const PairEval (&ev)[PPL], int b) {
                    float wsum = 0.f;
                    if (STATS) ++st_eval;
#pragma unroll
                    for (int q = 0; q < PPL; ++q) {
                        const PairEval& e = ev[q];
                        if (e.valid && !done[q]) {
                            const float Tn = T[q] * (1.0f - e.alpha);
                            if (Tn < GSR_T_STOP) {
                                done[q] = true;
                            } else {
                                const float wgt = e.alpha * T[q];
                                const float2 w2 = make_float2(wgt, wgt);
                                C01[q] = __ffma2_rn(make_float2(q2.x, q2.y), w2, C01[q]);
                                C2D[q] = __ffma2_rn(make_float2(q2.z, q1.w), w2, C2D[q]);
                                T[q] = Tn;
                                last[q] = pos0 + (uint32_t)b;
                                if (SCORE) wsum += wgt;
                                if (STATS) ++st_lanes;
                            }
                        }
                    }
                    if (SCORE) {
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) wsum += __shfl_xor_sync(0xffffffffu, wsum, o);
                        if (lane == 0 && wsum != 0.f) atomicAdd(score + __float_as_uint(q2.w), wsum);
                    }
                };
                while (mask) {
                    const int b = __ffs(mask) - 1;
                    mask &= mask - 1;
                    const float4* rp = sp + 3 * b;
                    const float4 q0 = rp[0], q1 = rp[1], q2 = rp[2];
                    // Two passing entries per trip: the record loads and exponent of the second are in flight
                    // while the first is evaluated (a warp issues in order, so this halves the dependent
                    // LDS -> FMA -> EX2 latency paid per entry on the longest tile, which bounds the kernel:
                    // profiles/r02_balance.md).  Same arithmetic and order per entry.
                    int bb[2];
                    float4 r0[2], r1[2], r2[2];
                    bb[0] = b; r0[0] = q0; r1[0] = q1; r2[0] = q2;
                    int have = 1;                                      // warp-uniform
#pragma unroll
                    for (int j = 1; j < 2; ++j) {
                        const bool more = mask != 0u;
                        bb[j] = more ? __ffs(mask) - 1 : b;
                        mask &= mask - 1;                              // 0 stays 0
                        have += more ? 1 : 0;
                        const float4* rj = sp + 3 * bb[j];
                        r0[j] = rj[0]; r1[j] = rj[1]; r2[j] = rj[2];
                    }
                    PairEval ev[2][PPL];
#pragma unroll
                    for (int j = 0; j < 2; ++j)
#pragma unroll
                        for (int q = 0; q < PPL; ++q)
                            ev[j][q] = eval_pair(r0[j].x, r0[j].y, r0[j].w, r1[j].x, r1[j].y, r1[j].z, X, Y[q]);
#pragma unroll
                    for (int j = 0; j < 2; ++j)
                        if (j < have) blend(r1[j], r2[j], ev[j], bb[j]);
                }
                all_done = true;
#pragma unroll
                for (int q = 0; q < PPL; ++q) all_done = all_done && done[q];
                if (__all_sync(0xffffffffu, all_done)) break;
            }
        }
        cp_async_wait<0>();   // never leave copies in flight across tiles (early-out case)

        const size_t plane = (size_t)Hs * W;
#pragma unroll
        for (int q = 0; q < PPL; ++q) {
            if (inside[q]) {
                const size_t pix = (size_t)(row0 + Yi + 4 * q) * W + Xi;
                out_color[pix] = fmaf(T[q], bg0, C01[q].x);
                out_color[plane + pix] = fmaf(T[q], bg1, C01[q].y);
                out_color[2 * plane + pix] = fmaf(T[q], bg2, C2D[q].x);
                out_depth_alpha[pix] = C2D[q].y;
                out_depth_alpha[plane + pix] = T[q];
                n_contrib[pix] = last[q];
            }
            // this 8x4 block's entry in the backward's work lists (fwd block blk, pixel row set q)
            const uint32_t nb = __reduce_max_sync(0xffffffffu, last[q]);
            if (lane == 0) bwd_item_append(bwd_fill, bwd_items, ntiles, tile, ((blk >> 1) * PPL + q) * 2 + (blk & 1), nb);
        }
    }
    if (STATS && stats != nullptr) {
        const unsigned int tl = __reduce_add_sync(0xffffffffu, st_lanes);
        if (lane == 0) {
            atomicAdd(stats + GSR_STAT_FWD_EVAL, (unsigned long long)st_eval);
            atomicAdd(stats + GSR_STAT_FWD_LANES, (unsigned long long)tl);
        }
        if (threadIdx.x == 0) {
            const unsigned long long t1 = gsr_now_ns();
            atomicAdd(stats + GSR_STAT_FWD_BUSY, t1 - st_t0);
            atomicMax(stats + GSR_STAT_FWD_END, t1);
            atomicMax(stats + GSR_STAT_FWD_NBEGIN, ~st_t0);
            atomicAdd(stats + GSR_STAT_FWD_WORKERS, 1ull);
            atomicMax(stats + GSR_STAT_FWD_MAX_ITEM, st_max_item_ns);
        }
    }
}

// =============================================================================================
// Backward.  The kernel is called composite_bwd2 because it replaced round 1's composite_bwd;
// the profiling tools and the records in profiles/ know it by that name.  Per-(warp, Gaussian) body:
//   * branch-free: non-contributing lanes run the same arithmetic with alpha = G = 0 instead of a
//     divergent block + ten zero-initialisations (BSSY/BSYNC, 8 moves gone);
//   * packed fp32 (fma.rn.f32x2 / mul / add -> FFMA2, FMUL2, FADD2): the four channel-parallel
//     streams (r, g, b, depth) and the (x, y) geometry pairs go two per instruction, halving the
//     fma-pipe occupancy of the body (the fma pipe retires a 3-register FFMA every 2 cycles/SMSP);
//   * STATS instantiation counts evaluated / contributing (warp, Gaussian) pairs and the popcount
//     histogram for the secondary (pair-evaluation) roofline in bench.py; never timed.
// =============================================================================================
__device__ __forceinline__ int bwd_value_index(int lane) {
    // which of the 10 values this lane ends up owning (-1: a padding slot)
    int base = 0, n = 10;
    if (lane & 16) { base += 5; n = 5; } else { n = 5; }
    if (lane & 8) { base += 3; n = n - 3; } else { n = min(n, 3); }
    if (lane & 4) { base += 2; n = max(n - 2, 0); } else { n = min(n, 2); }
    if (lane & 2) { base += 1; n = max(n - 1, 0); } else { n = min(n, 1); }
    return n >= 1 ? base : -1;
}

// Halving butterfly: after the four calls and one last shuffle, lane L holds the warp-wide sum of value
// `vidx(L)` (see bwd_value_index); 5+3+2+1+1 = 12 shuffles for 10 values.  The selects are per register,
// the ADDs go in packed pairs.
template <int N, int XOR>
__device__ __forceinline__ void halve2(float (&v)[10], bool hi) {
    constexpr int Hh = (N + 1) / 2;
    float keep[Hh], recv[Hh];
#pragma unroll
    for (int k = 0; k < Hh; ++k) {
        const float lo = v[k];
        const float hv = (Hh + k < N) ? v[Hh + k] : 0.0f;
        const float send = hi ? lo : hv;
        keep[k] = hi ? hv : lo;
        recv[k] = __shfl_xor_sync(0xffffffffu, send, XOR);
    }
#pragma unroll
    for (int k = 0; k + 1 < Hh; k += 2) {
        const float2 r = __fadd2_rn(make_float2(keep[k], keep[k + 1]), make_float2(recv[k], recv[k + 1]));
        v[k] = r.x; v[k + 1] = r.y;
    }
    if (Hh & 1) v[Hh - 1] = keep[Hh - 1] + recv[Hh - 1];
}


template <bool STATS>
__global__ void __launch_bounds__(kWarps * 32, kMinCtas)
composite_bwd2_kernel(int H, int W, int gx, int gy_view, int Hs, int ntiles, const uint32_t* __restrict__ header,
                      const uint32_t* __restrict__ work_order,
                      const uint32_t* __restrict__ tile_start,
                      const unsigned long long* __restrict__ keys, const GsrRec* __restrict__ geom,
                      const float* __restrict__ bg, uint32_t* __restrict__ queue,
                      const float* __restrict__ out_depth_alpha,
                      const uint32_t* __restrict__ n_contrib, const float* __restrict__ dL_dcolor,
                      const float* __restrict__ dL_ddepth_alpha, float* __restrict__ dgeom,
                      unsigned long long* __restrict__ stats, const uint32_t* __restrict__ bwd_items) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    SmemRing& sm = *reinterpret_cast<SmemRing*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    GsrRec (*ring)[32] = sm.rec[wid];
    const uint32_t max_pairs = header[GSR_H_MAX_PAIRS];
    // Work lists written by the forward: (tile, block) items by size class of the consumed list length.
    // Lane l holds the END of class (31 - l) in the concatenated longest-first order.
    uint32_t cls_end = header[GSR_H_BWD_FILL + (GSR_BWD_CLASSES - 1 - lane)];
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, cls_end, o);
        if (lane >= o) cls_end += t;
    }
    const uint32_t num_items = __shfl_sync(0xffffffffu, cls_end, 31);
    const size_t cls_cap = (size_t)ntiles * 8;
    static_assert(kWarps % GSR_NQUEUE == 0, "static first items must end on a sub-queue boundary");
    const uint32_t nworkers = gridDim.x * kWarps;            // the first item of every warp is static: no atomic
    const uint32_t i_first = (nworkers + GSR_NQUEUE - 1) / GSR_NQUEUE;
    bool first_item = true;
    const int vidx = bwd_value_index(lane);
    const bool commit_lane = (vidx >= 0) && !(lane & 1);
    const size_t plane = (size_t)Hs * W;
    unsigned long long st_eval = 0, st_contrib = 0, st_lanes = 0;
    unsigned long long st_hist[6] = {0, 0, 0, 0, 0, 0};
    unsigned long long st_t0 = 0, st_item_eval0 = 0, st_item_t0 = 0, st_max_item = 0, st_max_item_ns = 0;
    if (STATS) st_t0 = gsr_now_ns();

    uint32_t qsel = (blockIdx.x * kWarps + wid) % GSR_NQUEUE, qtried = 0;
    for (;;) {
        if (STATS) {
            if (st_eval - st_item_eval0 > st_max_item) st_max_item = st_eval - st_item_eval0;
            const unsigned long long t = gsr_now_ns();
            if (st_item_t0 && t - st_item_t0 > st_max_item_ns) st_max_item_ns = t - st_item_t0;
            st_item_eval0 = st_eval; st_item_t0 = t;
        }
        // position w in the longest-first order: warp g starts with w = g, later ones come from the split queue
        uint32_t w;
        if (first_item) {
            first_item = false;
            w = blockIdx.x * kWarps + wid;
            if (w >= num_items) break;
        } else {
            uint32_t i = 0xffffffffu;
            if (lane == 0) {
                while (qtried < GSR_NQUEUE) {
                    const uint32_t cand = (atomicAdd(queue + qsel, 1u) + i_first) * GSR_NQUEUE + qsel;
                    if (cand < num_items) { i = cand; break; }
                    qsel = (qsel + 1) % GSR_NQUEUE;
                    ++qtried;
                }
            }
            w = __shfl_sync(0xffffffffu, i, 0);
            if (w == 0xffffffffu) break;
        }
        const int cdone = __popc(__ballot_sync(0xffffffffu, cls_end <= w));          // classes entirely before w
        const uint32_t cstart = __shfl_sync(0xffffffffu, cls_end, (cdone + 31) & 31);
        const uint32_t item = __ldg(bwd_items + (size_t)(GSR_BWD_CLASSES - 1 - cdone) * cls_cap + (w - (cdone ? cstart : 0u)));
        const uint32_t tile = item >> 3;
        const int blk = (int)(item & 7u);
        uint32_t beg = tile_start[tile], end = tile_start[tile + 1];
        if (end > max_pairs) end = max_pairs;
        if (beg > end) beg = end;
        const unsigned long long* tk = keys + beg;
        const int tys = tile / gx, txi = tile - tys * gx;
        const int view = tys / gy_view, tyi = tys - view * gy_view;      // view-local evaluation, stacked addressing
        const int row0 = view * gy_view * GSR_TILE;
        const float* bgv = bg + 3 * view;
        const float bg0 = __ldg(bgv), bg1 = __ldg(bgv + 1), bg2 = __ldg(bgv + 2);
        const int X0i = txi * GSR_TILE + (blk & 1) * 8, Y0i = tyi * GSR_TILE + (blk >> 1) * 4;
        const int Xi = X0i + (lane & 7), Yi = Y0i + (lane >> 3);
        const float X0 = (float)X0i, Y0 = (float)Y0i;
        const float2 XY = make_float2(-(float)Xi, -(float)Yi);
        uint32_t last = 0;
        float Tfinal = 1.f, dT = 0.f;
        float2 dC01 = make_float2(0.f, 0.f), dC2D = make_float2(0.f, 0.f);
        if (Xi < W && Yi < H) {
            const size_t pix = (size_t)(row0 + Yi) * W + Xi;
            last = n_contrib[pix];
            Tfinal = out_depth_alpha[plane + pix];
            dC01.x = dL_dcolor[pix]; dC01.y = dL_dcolor[plane + pix]; dC2D.x = dL_dcolor[2 * plane + pix];
            dC2D.y = dL_ddepth_alpha[pix]; dT = dL_ddepth_alpha[plane + pix];
        }
        if ((int)last > (int)(end - beg)) last = end - beg;   // overflow safety
        const int n = (int)__reduce_max_sync(0xffffffffu, last);   // only entries [0, n) reached this block
        const int nsub = (n + 31) >> 5;
        const float bgT = Tfinal * (bg0 * dC01.x + bg1 * dC01.y + bg2 * dC2D.x + dT);   // Tfinal * bgterm
        float T = Tfinal;
        float2 acc01 = make_float2(0.f, 0.f), acc2D = make_float2(0.f, 0.f);

        // sub-chunks are visited from the back: visit v <-> sub-chunk nsub-1-v
        unsigned long long kq0, kq1;
        {
            unsigned long long kk[kSlots + 1];
#pragma unroll
            for (int j = 0; j < kSlots + 1; ++j) {
                const int e = (nsub - 1 - j) * 32 + lane;
                kk[j] = (j < nsub && e < n) ? __ldg(tk + e) : 0ull;
            }
#pragma unroll
            for (int j = 0; j < kSlots - 1; ++j) {
                const int e = (nsub - 1 - j) * 32 + lane;
                if (j < nsub && e < n) gather_record(&ring[j][lane], geom, kk[j]);
                cp_async_commit();
            }
            kq0 = kk[kSlots - 1]; kq1 = kk[kSlots];
        }
        for (int v = 0; v < nsub; ++v) {
            {
                const int g = v + kSlots - 1;
                if (g < nsub) gather_record(&ring[g % kSlots][lane], geom, kq0);   // earlier sub-chunks are full
                cp_async_commit();
                kq0 = kq1;
                const int g2 = v + kSlots + 1;
                kq1 = (g2 < nsub) ? __ldg(tk + (nsub - 1 - g2) * 32 + lane) : 0ull;
            }
            cp_async_wait<kSlots - 1>();
            __syncwarp();
            const GsrRec* st = ring[v % kSlots];
            const int sidx = nsub - 1 - v;
            const int cnt = min(32, n - sidx * 32);
            bool pass = false;
            if (lane < cnt) {
                const float4 q0 = *reinterpret_cast<const float4*>(&st[lane]);
                pass = cull_pass(q0.x, q0.y, __float_as_uint(q0.z), X0, Y0);
            }
            uint32_t mask = __ballot_sync(0xffffffffu, pass);
            const float4* sp = reinterpret_cast<const float4*>(st);
            const uint32_t pos0 = (uint32_t)(sidx * 32 + 1);
            while (mask) {
                const int b = 31 - __clz(mask);
                mask &= ~(1u << b);
                const float4* rp = sp + 3 * b;
                const float4 q0 = rp[0], q1 = rp[1];
                const uint32_t pos = pos0 + (uint32_t)b;
                // ---- the blending test (identical decisions to eval_pair) ----
                const float2 d = __fadd2_rn(make_float2(q0.x, q0.y), XY);          // (dx, dy)
#ifdef GSR_EXACT_EXP
                const PairEval e = eval_pair(q0.x, q0.y, q0.w, q1.x, q1.y, q1.z, -XY.x, -XY.y);
                const float G = e.G, alpha = e.alpha;
                const bool valid = e.valid;
#else
                const float u = __fmaf_rn(q0.w, d.x, __fmul_rn(q1.x, d.y));
                const float p2 = __fmaf_rn(__fmul_rn(q1.y, d.y), d.y, __fmul_rn(u, d.x));
                const float G = ex2_approx(p2);
                const float alpha = fminf(GSR_ALPHA_MAX, __fmul_rn(q1.z, G));
                const bool valid = (p2 <= 0.0f) && (alpha >= GSR_ALPHA_MIN);
#endif
                const bool contrib = valid && pos <= last;
                const uint32_t cm = __ballot_sync(0xffffffffu, contrib);
                if (STATS) ++st_eval;
                if (cm == 0u) continue;
                const float4 q2 = rp[2];
                // ---- branch-free body: non-contributing lanes carry alpha = G = 0 ----
                const float am = contrib ? alpha : 0.0f;
                const float Gm = contrib ? G : 0.0f;
                const float rom = rcp_approx(1.0f - am);
                T = contrib ? T * rom : T;                       // transmittance in front of this entry
                const float wgt = am * T;
                const float2 c01 = make_float2(q2.x, q2.y), c2D = make_float2(q2.z, q1.w);
                const float2 nacc01 = make_float2(-acc01.x, -acc01.y), nacc2D = make_float2(-acc2D.x, -acc2D.y);
                const float2 d01 = __fadd2_rn(c01, nacc01), d2D = __fadd2_rn(c2D, nacc2D);
                const float2 dot2 = __ffma2_rn(d2D, dC2D, __fmul2_rn(d01, dC01));
                const float dLda = (dot2.x + dot2.y) * T - bgT * rom;
                const float2 am2 = make_float2(am, am);
                acc01 = __ffma2_rn(am2, d01, acc01);
                acc2D = __ffma2_rn(am2, d2D, acc2D);
                float vv[10];
                vv[5] = Gm * dLda;
                const float gG = q1.z * vv[5];                   // dL/dG * G (no zeroing under the 0.99 clamp)
#ifdef GSR_EXACT_EXP
                const float2 gs = make_float2(-(q0.w * d.x + q1.x * d.y), -(q1.y * d.y + q1.x * d.x));
#else
                const float2 gs = __ffma2_rn(make_float2(q0.w + q0.w, q1.y + q1.y), d, __fmul2_rn(make_float2(q1.x, q1.x), make_float2(d.y, d.x)));
#endif
                const float2 gG2 = make_float2(gG, gG);
                const float2 v01 = __fmul2_rn(gG2, gs);
                const float2 tu = __fmul2_rn(gG2, d);             // (gG dx, gG dy)
                const float2 v24 = __fmul2_rn(tu, d);             // (gG dx^2, gG dy^2)
                vv[0] = v01.x; vv[1] = v01.y; vv[2] = v24.x; vv[3] = tu.x * d.y; vv[4] = v24.y;
                const float2 w2 = make_float2(wgt, wgt);
                const float2 v67 = __fmul2_rn(w2, dC01), v89 = __fmul2_rn(w2, dC2D);
                vv[6] = v67.x; vv[7] = v67.y; vv[8] = v89.x; vv[9] = v89.y;
                float* row = dgeom + 12 * (size_t)__float_as_uint(q2.w);
                if (STATS) {
                    const int k = __popc(cm);
                    ++st_contrib; st_lanes += k;
                    ++st_hist[k == 1 ? 0 : k == 2 ? 1 : k <= 4 ? 2 : k <= 8 ? 3 : k <= 16 ? 4 : 5];
                }
                halve2<10, 16>(vv, lane & 16);
                halve2<5, 8>(vv, lane & 8);
                halve2<3, 4>(vv, lane & 4);
                halve2<2, 2>(vv, lane & 2);
                const float tot = vv[0] + __shfl_xor_sync(0xffffffffu, vv[0], 1);
                if (commit_lane) atomicAdd(row + vidx, tot);
            }
            __syncwarp();
        }
        cp_async_wait<0>();
        __syncwarp();
    }
    if (STATS && lane == 0 && stats != nullptr) {
        atomicAdd(stats + GSR_STAT_BWD_EVAL, st_eval);
        atomicAdd(stats + GSR_STAT_BWD_CONTRIB, st_contrib);
        atomicAdd(stats + GSR_STAT_BWD_LANES, st_lanes);
#pragma unroll
        for (int j = 0; j < 6; ++j) atomicAdd(stats + GSR_STAT_BWD_HIST + j, st_hist[j]);
        const unsigned long long t1 = gsr_now_ns();
        atomicAdd(stats + GSR_STAT_BWD_BUSY, t1 - st_t0);
        atomicMax(stats + GSR_STAT_BWD_END, t1);
        atomicMax(stats + GSR_STAT_BWD_NBEGIN, ~st_t0);
        atomicAdd(stats + GSR_STAT_BWD_WORKERS, 1ull);
        atomicMax(stats + GSR_STAT_BWD_MAX_ITEM, st_max_item);
        atomicMax(stats + GSR_STAT_BWD_MAX_ITEM_NS, st_max_item_ns);
    }
}

}  // namespace

struct CompPtrs {
    GsrTileGrid grid;
    int H;                 // height of the (stacked) image the kernels render
    const uint32_t *header, *tile_start, *work_order;
    const unsigned long long* keys;
    const GsrRec* geom;
    uint32_t* n_contrib;
    uint32_t *bwd_fill, *bwd_items;   // backward work lists (items == nullptr: the forward was issued without backward)
};
static CompPtrs comp_ptrs(const uint8_t* saved, const b200gsr_saved_layout& vl, int H, int W, int num_views, int gy_view) {
    CompPtrs c;
    c.grid = gsr_grid(H, W);
    c.H = H;
    if (num_views > 1) {   // views stacked vertically, each padded to whole tile rows
        c.grid.gy = num_views * gy_view; c.grid.ntiles = c.grid.gx * c.grid.gy;
        c.H = c.grid.gy * GSR_TILE;
    }
    c.header = reinterpret_cast<const uint32_t*>(saved + vl.header);
    c.tile_start = reinterpret_cast<const uint32_t*>(saved + vl.tile_start);
    c.work_order = reinterpret_cast<const uint32_t*>(saved + vl.work_order);
    c.keys = reinterpret_cast<const unsigned long long*>(saved + vl.keys);
    c.geom = reinterpret_cast<const GsrRec*>(saved + vl.geom);
    c.n_contrib = reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(saved) + vl.n_contrib);
    c.bwd_fill = reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(saved) + vl.header) + GSR_H_BWD_FILL;
    c.bwd_items = vl.bwd_items < vl.total ? reinterpret_cast<uint32_t*>(const_cast<uint8_t*>(saved) + vl.bwd_items) : nullptr;
    return c;
}

template <bool SCORE, bool STATS>
static cudaError_t launch_fwd(const GsrFwdArgs& a, int nblocks, const CompPtrs& c, uint32_t* queue) {
    const int smem = (int)sizeof(SmemCta);
    static std::atomic<unsigned long long> attr_done{0};
    cudaError_t e = gsr_smem_once(composite_fwd_kernel<SCORE, 1, STATS>, smem, attr_done);
    if (e != cudaSuccess) return e;
    composite_fwd_kernel<SCORE, 1, STATS><<<nblocks, 256, smem, a.stream>>>(
        a.prm.image_height, a.prm.image_width, c.grid.gx, a.gy_view, c.H, c.grid.ntiles, c.header, c.work_order, c.tile_start,
        c.keys, c.geom, a.prm.bg, queue, a.out_color, a.out_depth_alpha, c.n_contrib, a.score, a.stats, c.bwd_fill, c.bwd_items);
    return cudaGetLastError();
}

cudaError_t gsr_launch_composite_fwd(const GsrFwdArgs& a) {
    const CompPtrs c = comp_ptrs(a.saved, a.vl, a.prm.image_height, a.prm.image_width, a.num_views, a.gy_view);
    if (c.grid.ntiles == 0) return cudaSuccess;
    uint32_t* queue = reinterpret_cast<uint32_t*>(a.scratch + a.sl.counters) + GSR_C_FWD_QUEUE;
    const int nblocks = min(c.grid.ntiles, a.num_sms * 6);
    if (a.stats != nullptr)
        return a.prm.score_flag ? launch_fwd<true, true>(a, nblocks, c, queue)
                                : launch_fwd<false, true>(a, nblocks, c, queue);
    return a.prm.score_flag ? launch_fwd<true, false>(a, nblocks, c, queue)
                            : launch_fwd<false, false>(a, nblocks, c, queue);
}

template <bool STATS>
static cudaError_t launch_bwd(const GsrBwdArgs& a, const CompPtrs& c, uint32_t* queue, float* dgeom) {
    const int smem = (int)sizeof(SmemRing);
    const int nblocks = min(c.grid.ntiles, a.num_sms * kMinCtas);
    static std::atomic<unsigned long long> attr_done{0};
    cudaError_t e = gsr_smem_once(composite_bwd2_kernel<STATS>, smem, attr_done);
    if (e != cudaSuccess) return e;
    composite_bwd2_kernel<STATS><<<nblocks, kWarps * 32, smem, a.stream>>>(
        a.prm.image_height, a.prm.image_width, c.grid.gx, a.gy_view, c.H, c.grid.ntiles, c.header, c.work_order, c.tile_start,
        c.keys, c.geom, a.prm.bg, queue, a.out_depth_alpha, c.n_contrib, a.dL_dcolor, a.dL_ddepth_alpha, dgeom,
        a.stats, c.bwd_items);
    return cudaGetLastError();
}

cudaError_t gsr_launch_composite_bwd(const GsrBwdArgs& a) {
    const CompPtrs c = comp_ptrs(a.saved, a.vl, a.prm.image_height, a.prm.image_width, a.num_views, a.gy_view);
    if (c.grid.ntiles == 0) return cudaSuccess;
    uint32_t* queue = reinterpret_cast<uint32_t*>(a.saved + a.vl.header) + GSR_H_BWD_QUEUE;
    float* dgeom = reinterpret_cast<float*>(a.saved + a.vl.dgeom);
    return a.stats != nullptr ? launch_bwd<true>(a, c, queue, dgeom) : launch_bwd<false>(a, c, queue, dgeom);
}
