// Shared device-side definitions for the B200 (sm_100a) Gaussian rasterizer kernels.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>

#include "../../include/b200gsr.h"

#define GSR_TILE 16
#define GSR_NEAR_Z 0.2f
#define GSR_ALPHA_MIN (1.0f / 255.0f)
#define GSR_ALPHA_MAX 0.99f
#define GSR_T_STOP 1e-4f
#define GSR_LOG2E 1.4426950408889634f
#define GSR_LN2 0.6931471805599453f

// One (tile, Gaussian) pair as consumed by the composite kernels; also the per-Gaussian
// "geom" record written by project_sh (the sort epilogue copies geom[idx] -> sorted[pos]).
// 48 bytes = 3 x 16 B, so 8 consecutive lanes reading one 16-B part each hit 8 distinct
// 4-bank groups (stride 12 words) -> conflict-free LDS.128, and a record moves as three
// 16-byte cp.async copies.
struct __align__(16) GsrRec {
    // part 0: everything the per-warp cull test needs
    float px, py;   // pixel-space mean
    uint32_t ext;   // half2 (ext_x, ext_y): conservative half extents of {alpha >= 1/255}
    float A;        // scaled conic: log2(G) = A*dx*dx + B*dx*dy + C*dy*dy  (GSR_EXACT_EXP: raw conic.x)
    // part 1
    float B, C;     //   A = -0.5*log2e*conic.x, B = -log2e*conic.y, C = -0.5*log2e*conic.z
    float opacity;
    float depth;    // view-space z
    // part 2
    float r, g, b;  // colour (SH evaluated, +0.5, clamped >= 0) or colors_precomp
    uint32_t idx;   // Gaussian index
};
static_assert(sizeof(GsrRec) == 48, "record must be 48 bytes");

struct GsrTileGrid {
    int gx, gy, ntiles;
};

__host__ __device__ inline GsrTileGrid gsr_grid(int H, int W) {
    GsrTileGrid g;
    g.gx = (W + GSR_TILE - 1) / GSR_TILE;
    g.gy = (H + GSR_TILE - 1) / GSR_TILE;
    g.ntiles = g.gx * g.gy;
    return g;
}

// header words in the saved buffer (uint32[GSR_H_WORDS])
enum { GSR_H_NUM_PAIRS = 0, GSR_H_MAX_PAIRS = 1, GSR_H_NUM_TILES = 2, GSR_H_OVERFLOW = 3,
       GSR_H_NUM_BIG = 4, GSR_H_NUM_NONEMPTY = 5,
       GSR_H_BWD_QUEUE = 8,       // [8, 8+GSR_NQUEUE): work-queue counters of composite_bwd; zeroed by the
                                  // forward's scan kernel and restored to zero by project_bwd, so a saved
                                  // buffer can be back-propagated any number of times without a memset
       GSR_H_BWD_FILL = 32,       // [32, 64): items per size class of the backward's work lists (written by the
                                  // forward's composite kernel, zeroed by its scan kernel)
       GSR_H_WORDS = 64 };
// Backward work items = (tile, 8x4-pixel block) pairs that blended at least one entry, binned by the
// forward into GSR_BWD_CLASSES size classes of the block's consumed list length (two classes per power
// of two); the backward pops the longest first.  List of class k: bwd_items[k * num_tiles * 8 ...].
#define GSR_BWD_CLASSES 32
__host__ __device__ inline int gsr_bwd_class(uint32_t n) {     // n >= 1
#ifdef __CUDA_ARCH__
    const int e = 31 - __clz((int)n);
#else
    int e = 0; while (e < 31 && (n >> (e + 1)) != 0u) ++e;
#endif
    const int k = 2 * e + (e > 0 ? (int)((n >> (e - 1)) & 1u) : 0);
    return k < GSR_BWD_CLASSES - 1 ? k : GSR_BWD_CLASSES - 1;
}
// counters in scratch
// The tile work queue is split into GSR_NQUEUE sub-queues (tile w lives in queue w % NQUEUE): one
// shared counter would serialise every fetch at the ~30 ns same-address L2 atomic rate.
#define GSR_NQUEUE 8
#define GSR_NCOUNTERS 128
enum { GSR_C_FWD_QUEUE = 0 };

#define GSR_SORT_SMALL_MAX 4096   // keys sorted by the 256-thread kernel (256 x 16 items)
#define GSR_SORT_BIG_CHUNK 16384  // keys per smem chunk of the 1024-thread kernel (1024 x 16 items)
// Tile counters/cursors are privatised into GSR_COPIES arrays (copy = (gaussian_idx>>5) & mask):
// same-address L2 atomics serialise at ~30 ns each, so the hottest tile bounds the kernel.
#define GSR_COPIES 16
// Block-multisplit binning (default when the tile grid fits in shared memory): a CTA of 1024
// threads owns GSR_MS_ITEMS*1024 consecutive Gaussians and histograms their tile hits in smem, so
// global atomics drop from one per (Gaussian, tile) pair to one per (CTA, touched tile).
#define GSR_MS_ITEMS 4
// Number of multisplit CTAs for P (virtual) Gaussians: at most 4096 Gaussians per CTA; a scene that
// would fill less than one wave (2 CTAs x 148 SMs) is spread over the whole wave instead, down to 256
// Gaussians per CTA, so that every SM carries the same load.
#define GSR_MS_WAVE_CTAS 296
__host__ __device__ inline int gsr_ms_blocks(long long P) {
    const long long full = (P + 1024 * GSR_MS_ITEMS - 1) / (1024 * GSR_MS_ITEMS);
    if (full >= GSR_MS_WAVE_CTAS) return (int)full;
    const long long fine = (P + 255) / 256;
    return (int)(fine < 1 ? 1 : (fine < GSR_MS_WAVE_CTAS ? fine : GSR_MS_WAVE_CTAS));
}
#define GSR_MS_MAX_TILES 12288   // 4 B x tiles of dynamic smem (48 KB); 12 tiles per thread in the scan kernel
__host__ __device__ inline bool gsr_use_multisplit(int ntiles) { return ntiles <= GSR_MS_MAX_TILES; }

#ifdef __CUDACC__
// ---- 128-bit global access helpers -------------------------------------------------------
__device__ __forceinline__ float4 ldg_f4(const void* p) {
    return *reinterpret_cast<const float4*>(p);
}
__device__ __forceinline__ void stg_na_f4(void* p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};"
                 :: "l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
// Default build: exp via ONE MUFU (ex2.approx on a conic pre-scaled by log2 e), T recovery in the
// backward via rcp.approx.  -DGSR_EXACT_EXP builds the parity-diagnostic variant
// (libb200gsr_exact.so): the record keeps the UNSCALED conic, the exponent is evaluated with
// individually rounded fp32 ops in the oracle's operation order (oracle/splat_ref.py::composite),
// exp is expf() and the reciprocal an IEEE division.  It exists to show that the forward outliers
// against the oracle are exp-approximation artefacts at the discontinuous 1/255 and 1e-4 tests
// (profiles/r02_parity_stats.json) and what the approximation buys (ms).
#ifdef GSR_EXACT_EXP
#define GSR_PX_GRAD_SCALE 1.0f
__device__ __forceinline__ float rcp_approx(float x) { return __fdiv_rn(1.0f, x); }
#else
#define GSR_PX_GRAD_SCALE GSR_LN2
__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
    float y;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}
#endif

// ---- shared-memory address helper (cp.async destinations) ----------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}
#endif  // __CUDACC__

// ---- kernel launchers (defined in the .cu files, called from api.cu) ---------------------
struct GsrFwdArgs {
    b200gsr_params prm;
    const float *means3D, *shs, *colors, *opac, *scales, *rots, *cov3d;
    float *out_color, *out_depth_alpha, *score;
    int32_t* radii;
    uint8_t *scratch, *saved;
    b200gsr_scratch_layout sl;
    b200gsr_saved_layout vl;
    uint32_t max_pairs;
    uint32_t* host_notify;
    uint32_t notify_seq;
    uint32_t flags;        // B200GSR_FWD_*
    // multi-view (b200gsr_forward_views): the views are stacked vertically into one image of
    // num_views * gy_view tile rows; view v's Gaussians are the virtual Gaussians [v*P_view, (v+1)*P_view).
    // Single-view calls: view = 0, num_views = 1, P_view = prm.P, gy_view = tile rows of the image.
    int view, num_views, P_view, gy_view;
    int num_sms;           // of the current device (cached per device in api.cu)
    unsigned long long* stats;
    cudaStream_t stream;
};

struct GsrBwdArgs {
    b200gsr_params prm;
    const float *means3D, *shs, *colors, *opac, *scales, *rots, *cov3d;
    const int32_t* radii;
    const float *out_depth_alpha, *dL_dcolor, *dL_ddepth_alpha;
    uint8_t* saved;     // counters + gradient accumulators inside are consumed and restored
    uint8_t* scratch;   // unused (kept for layout symmetry)
    b200gsr_scratch_layout sl;
    b200gsr_saved_layout vl;
    uint32_t max_pairs;
    float *d_means3D, *d_means2D, *d_shs, *d_colors, *d_opac, *d_scales, *d_rots, *d_cov3d;
    int view, num_views, P_view, gy_view;   // see GsrFwdArgs
    int accumulate;        // project_bwd adds into the gradient outputs instead of overwriting (views sharing a parameter)
    int dsh_coefs;         // coefficients per row of d_shs (0 = M, the reference layout)
    int num_sms;
    unsigned long long* stats;   // optional device counters (b200gsr_debug_counters); selects the STATS kernels
    cudaStream_t stream;
};

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) once per (kernel, device) instead of on every
// launch: `done` is a per-call-site bit mask indexed by device ordinal.
template <typename F>
inline cudaError_t gsr_smem_once(F func, int bytes, std::atomic<unsigned long long>& done) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    const unsigned long long bit = 1ull << (dev & 63);
    if (done.load(std::memory_order_acquire) & bit) return cudaSuccess;
    e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) done.fetch_or(bit, std::memory_order_release);
    return e;
}

cudaError_t gsr_launch_project(const GsrFwdArgs& a);
cudaError_t gsr_launch_count(const GsrFwdArgs& a);         // multisplit path: per-tile pair counts
cudaError_t gsr_launch_scan(const GsrFwdArgs& a);          // exclusive scan + work order + host notify
cudaError_t gsr_launch_scatter(const GsrFwdArgs& a);       // append keys to tile lists
cudaError_t gsr_launch_sort(const GsrFwdArgs& a, cudaStream_t side, cudaEvent_t fork, cudaEvent_t join);   // per-tile sort (2 kernels, concurrent when `side` is given)
cudaError_t gsr_launch_composite_fwd(const GsrFwdArgs& a);
cudaError_t gsr_launch_composite_bwd(const GsrBwdArgs& a);
cudaError_t gsr_launch_project_bwd(const GsrBwdArgs& a);
cudaError_t gsr_launch_sh_grad_expand(int P, int M, int deg, int nviews, const float* means3D, const float* dcol,
                                      size_t stride, float* d_shs, cudaStream_t s);
cudaError_t gsr_launch_mark_visible(int P, const float* means3D, const float* view,
                                    const float* proj, uint8_t* visible, cudaStream_t s);

// scene assembly (assemble.cu)
cudaError_t gsr_launch_assemble(bool backward, int num_groups, const b200gsr_group* groups,
                                const b200gsr_group_grad* grads, int M, int B, float c_shs, float c_scale,
                                const float* z_shs, const float* z_scales, unsigned long long seed,
                                float* means3D, float* opac, float* scales, float* rots, float* shs, cudaStream_t s);

// disparity post-processing (postprocess.cu)
cudaError_t gsr_launch_disparity_fwd(int B, int N, const float* da, const float* focal, float* out, void* stats,
                                     int num_sms, cudaStream_t s);
cudaError_t gsr_launch_disparity_bwd(int B, int N, const float* da, const float* focal, const float* g_out,
                                     const float* g_alpha, void* stats, float* d_da, int num_sms, cudaStream_t s);

// densification / pruning (densify.cu)
cudaError_t gsr_densify_stats(int P, const float* vs_grad, const int32_t* radii, float* accum, float* denom,
                              float* max_radii, cudaStream_t s);
size_t gsr_densify_scratch_bytes(int P);
cudaError_t gsr_densify_plan(int P, const float* accum, const float* denom, const float* scaling, const float* opacity,
                             float max_grad, float dense_extent, float min_opacity, float big_ws, float child_div, void* scratch,
                             uint32_t* totals5, cudaStream_t s);
cudaError_t gsr_densify_map(int P, int N, const void* scratch, const uint32_t* totals5, int32_t* src_map,
                            int32_t* child_draw, cudaStream_t s);
cudaError_t gsr_compact_plan(int P, const uint8_t* keep, void* scratch, int32_t* src_map, uint32_t* count, cudaStream_t s);
cudaError_t gsr_gather_rows(int n_out, int row_floats, const int32_t* src_map, const float* in, float* out,
                            int zero_appended, cudaStream_t s);
cudaError_t gsr_split_children(int n_out, int first_child, float child_div, const int32_t* src_map, const int32_t* child_draw,
                               const float* xyz, const float* scaling, const float* rotation, const float* z,
                               float* xyz_out, float* scaling_out, cudaStream_t s);
cudaError_t gsr_kth_smallest(int n, const float* v, uint32_t k, void* scratch, float* out, int num_sms, cudaStream_t s);

// simple_knn replacement (knn.cu)
size_t gsr_knn_scratch_bytes(int P, int* max_cells_out);
cudaError_t gsr_launch_knn(int P, const float* pts, float* out, uint8_t* scratch, cudaStream_t s);
