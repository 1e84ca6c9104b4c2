/*
 * b200gsr.h - C ABI of the B200-native differentiable 3D-Gaussian rasterizer.
 *
 * This is the drop-in boundary for the ONE native op DreamScene calls on its render path:
 * the un-vendored extension `diff_gaussian_rasterization._C`
 * (DreamScene-Project/comp-diff-gaussian-rasterization; /root/reference/README.md:47,50,
 * imported at /root/reference/scene_gaussian.py:11-12 and called at :637-646, :861-870,
 * :1012-1021).  Upstream exposes it through pybind as
 *     _C.rasterize_gaussians(...)            -> b200gsr_forward
 *     _C.rasterize_gaussians_backward(...)   -> b200gsr_backward
 *     _C.mark_visible(...)                   -> b200gsr_mark_visible (never called by DreamScene)
 * Here the same three entry points are plain `extern "C"` functions over raw device pointers
 * (no torch types), bound from Python with ctypes (dreamscene_b200/_lib.py) behind the
 * byte-compatible GaussianRasterizationSettings / GaussianRasterizer Python surface.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller unless stated otherwise;
 *     the library never allocates or frees device memory.  Process-wide state it does keep:
 *     a thread-local error string; per device, one lazily created non-blocking side stream +
 *     two events (lets the two tile-sort size classes overlap; creation is mutex-guarded, calls
 *     on DIFFERENT streams of one device from different host threads must still be serialised by
 *     the caller because they share those events); per kernel, a "shared-memory attribute set"
 *     bit per device; and the optional b200gsr_profile_* event store (not thread-safe);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*) of the CURRENT device;
 *     no host sync, no memset nodes on the main path (capturable into a CUDA graph);
 *   - return value: 0 = OK, negative = error (see b200gsr_last_error());
 *   - tensors are dense, row-major fp32 unless stated; layouts follow the reference call sites:
 *       means3D[P,3] means2D-grad[P,3] shs[P,M,3] colors_precomp[P,3] opacities[P,1]
 *       scales[P,3] rotations[P,4](w,x,y,z) cov3D_precomp[P,6](xx,xy,xz,yy,yz,zz)
 *       out_color[3,H,W] out_depth_alpha[2,H,W] radii[P](int32) score[P]
 *       viewmatrix/projmatrix[4,4] exactly as passed by scene_gaussian.py:586-599
 *       (row-vector convention, flat index 4*row+col).
 */
#ifndef B200GSR_H
#define B200GSR_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GSR_VERSION 4

/* error codes */
#define B200GSR_OK 0
#define B200GSR_ERR_BAD_ARG (-1)      /* null pointer / inconsistent optional inputs */
#define B200GSR_ERR_WORKSPACE (-2)    /* scratch/saved buffer too small for (P,H,W,max_pairs) */
#define B200GSR_ERR_CUDA (-3)         /* a CUDA runtime call or launch failed */
#define B200GSR_ERR_UNSUPPORTED (-4)  /* e.g. sh_degree > 3 */

/* Per-call constants == GaussianRasterizationSettings (scene_gaussian.py:586-599) + sizes. */
typedef struct b200gsr_params {
    int32_t P;               /* number of Gaussians */
    int32_t M;               /* SH coefficients per channel = (max_sh_degree+1)^2 (stride) */
    int32_t sh_degree;       /* active degree, 0..3, (sh_degree+1)^2 <= M */
    int32_t image_height;
    int32_t image_width;
    float tanfovx;
    float tanfovy;
    float scale_modifier;
    int32_t prefiltered;     /* accepted for API compatibility; ignored (as upstream's render path) */
    int32_t score_flag;      /* 1: also accumulate important_score[P] */
    const float* bg;         /* device [3] */
    const float* viewmatrix; /* device [16] */
    const float* projmatrix; /* device [16] */
    const float* campos;     /* device [3] */
} b200gsr_params;

/* Byte offsets of the arrays inside the `saved` buffer (for tests / debugging / backward). */
typedef struct b200gsr_saved_layout {
    size_t header;        /* uint32[64]: [0]=num_pairs (true D, may exceed max_pairs) [1]=max_pairs
                             [2]=num_tiles [3]=overflow flag [4]=num_big_tiles [5]=non-empty tiles
                             [8..15]=backward work-queue counters (zero between calls)
                             [32..63]=items per size class of bwd_items; rest reserved */
    size_t tile_start;    /* uint32[num_tiles+1] exclusive prefix of per-tile pair counts */
    size_t work_order;    /* uint32[num_tiles] tile ids, longest list first */
    size_t n_contrib;     /* uint32[H*W] index(1-based) of the last blended entry per pixel */
    size_t keys;          /* uint64[max_pairs+2] (depth_bits<<32 | gaussian idx), tile-major, depth-sorted */
    size_t geom;          /* 48-byte per-Gaussian records [P] (see common.cuh), gathered by the composite kernels */
    size_t dgeom;         /* float[P*12] screen-space gradient accumulators of the backward.  Rows of visible
                             Gaussians are zeroed by the forward and restored to zero by the backward
                             (read-and-clear), so no memset is ever needed.  Absent (size 0) when the
                             layout is queried with with_backward = 0 */
    size_t bwd_items;     /* uint32[32][num_tiles*8] work lists of the backward: (tile*8 + 8x4-pixel block) of
                             every block that blended an entry, by size class of its consumed list length
                             (written by the forward; longest class popped first).  Absent with
                             with_backward = 0 */
    size_t total;
} b200gsr_saved_layout;

/* Byte offsets inside the transient `scratch` buffer (valid until the next call on the stream). */
typedef struct b200gsr_scratch_layout {
    size_t counters;      /* uint32[128] split work-queue counters */
    size_t tile_count;    /* uint32[16][num_tiles] privatised per-tile pair counters */
    size_t tile_cursor;   /* uint32[16][num_tiles] write cursors */
    size_t rectdepth;     /* uint4[P]: (minx|miny<<16, maxx|maxy<<16, depth bits, tiles touched) */
    size_t ms_hist;       /* uint32[num_CTAs(P)][num_tiles] per-CTA tile histograms (multisplit binning) */
    size_t total;
} b200gsr_scratch_layout;

int b200gsr_version(void);
const char* b200gsr_last_error(void);

/* forward flags */
#define B200GSR_FWD_NO_BACKWARD 1u   /* `saved` was sized with with_backward = 0: skip the gradient accumulators */

/* Sizes/offsets of the two caller-owned buffers.  `saved` must stay alive until backward;
 * `scratch` is transient (forward only).  max_pairs = capacity for (tile,Gaussian) pairs
 * ("num_rendered").  with_backward = 0 drops the 48 B/Gaussian accumulator array (inference,
 * important_score renders). */
int b200gsr_saved_layout_query(int32_t P, int32_t H, int32_t W, uint64_t max_pairs,
                               int32_t with_backward, b200gsr_saved_layout* out);
int b200gsr_scratch_layout_query(int32_t P, int32_t H, int32_t W, uint64_t max_pairs,
                                 b200gsr_scratch_layout* out);

/*
 * Forward (replaces _C.rasterize_gaussians).  Exactly one of {shs, colors_precomp} and exactly
 * one of {(scales, rotations), cov3D_precomp} must be non-null (same rule the reference Python
 * enforces).  `score` may be null unless score_flag.  If the true pair count exceeds max_pairs the
 * kernels stay in bounds, header[3] is set and the images are INVALID: the caller reads header[0]
 * and re-issues the call with a larger capacity.  To learn the pair count without draining the
 * stream, pass `host_notify` = a pinned, device-mapped HOST buffer of 4 uint32: as soon as the
 * tile scan has run (long before compositing finishes) the device writes
 * {notify_seq, num_pairs, overflow, num_tiles} into it (system-scope fence, seq written last);
 * the host polls word 0.  Pass NULL to skip.
 */
int b200gsr_forward(const b200gsr_params* prm,
                    const float* means3D, const float* shs, const float* colors_precomp,
                    const float* opacities, const float* scales, const float* rotations,
                    const float* cov3D_precomp,
                    float* out_color, float* out_depth_alpha, int32_t* radii, float* score,
                    void* scratch, size_t scratch_bytes, void* saved, size_t saved_bytes,
                    uint64_t max_pairs, uint32_t flags, uint32_t* host_notify, uint32_t notify_seq,
                    void* stream);

/*
 * Backward (replaces _C.rasterize_gaussians_backward).  Inputs as in forward plus the forward's
 * radii / out_depth_alpha (channel 1 = final transmittance) / saved buffer and the incoming
 * gradients dL/dcolor[3,H,W], dL/ddepth_alpha[2,H,W].  Outputs are fully overwritten (zeros for
 * culled Gaussians): d_means3D[P,3], d_means2D[P,3] (NDC-scaled screen-space gradient, z=0),
 * d_opacities[P,1], and d_shs[P,M,3] | d_colors[P,3], (d_scales[P,3], d_rotations[P,4]) |
 * d_cov3D[P,6] matching the forward's input choice.  The call mutates and restores the
 * accumulators inside `saved` (hence non-const): the same `saved` may be back-propagated again
 * (retain_graph).  `scratch` is unused since version 2 (may be NULL / 0).
 */
int b200gsr_backward(const b200gsr_params* prm,
                     const float* means3D, const float* shs, const float* colors_precomp,
                     const float* opacities, const float* scales, const float* rotations,
                     const float* cov3D_precomp,
                     const int32_t* radii, const float* out_depth_alpha,
                     const float* dL_dcolor, const float* dL_ddepth_alpha,
                     void* saved, size_t saved_bytes, void* scratch, size_t scratch_bytes,
                     uint64_t max_pairs,
                     float* d_means3D, float* d_means2D, float* d_shs, float* d_colors,
                     float* d_opacities, float* d_scales, float* d_rotations, float* d_cov3D,
                     void* stream);

/*
 * Backward with a choice of SH gradient layout (additive; no upstream equivalent).  Same arguments as
 * b200gsr_backward plus
 *   dsh_coefs : 0 = d_shs has the reference layout [P, M, 3]; otherwise d_shs is a COMPACT
 *               [P, dsh_coefs, 3] array holding only the coefficients an active degree can touch
 *               ((sh_degree+1)^2 <= dsh_coefs <= M): the multi-GPU gradient payload at low degrees;
 *               -1 = FACTORED: d_shs is a [P, 3] array receiving dL/d(clamped colour).  The SH gradient of a
 *               view is the outer product basis(view direction) x that vector, so ranks exchange 3 floats per
 *               Gaussian and view instead of 3*M and rebuild the sum with b200gsr_sh_grad_expand.
 */
int b200gsr_backward_ex(const b200gsr_params* prm,
                        const float* means3D, const float* shs, const float* colors_precomp,
                        const float* opacities, const float* scales, const float* rotations,
                        const float* cov3D_precomp,
                        const int32_t* radii, const float* out_depth_alpha,
                        const float* dL_dcolor, const float* dL_ddepth_alpha,
                        void* saved, size_t saved_bytes, void* scratch, size_t scratch_bytes,
                        uint64_t max_pairs,
                        float* d_means3D, float* d_means2D, float* d_shs, float* d_colors,
                        float* d_opacities, float* d_scales, float* d_rotations, float* d_cov3D,
                        int32_t dsh_coefs, void* stream);

/*
 * Sum of the SH gradients of `num_views` views from their factored form (additive; multi-GPU view sharding):
 *   d_shs[i][k][c] = sum_v basis_k(normalize(means3D[i] - cam_v)) * dcol_v[i][c],  coefficients above sh_degree = 0.
 * View v's record starts at dcol + v * view_stride floats: [P][3] from b200gsr_backward_ex(dsh_coefs = -1), followed
 * by the view's camera centre (3 floats) - exactly what one all-gather of per-rank [3P + 3 (+pad)] buffers delivers.
 * The sum runs in view order, so every rank computes bit-identical gradients.  1 <= num_views <= 64.
 */
int b200gsr_sh_grad_expand(int32_t P, int32_t M, int32_t sh_degree, int32_t num_views, const float* means3D,
                           const float* dcol, size_t view_stride, float* d_shs, void* stream);

/*
 * Multi-view rendering (SURVEY.md 8 f1; additive, no upstream equivalent): B views of the same image
 * size and the same P in ONE tile-binning / sort / composite pass.  DreamScene renders C_batch_size = 4
 * views per training step one after the other (/root/reference/training/scene_trainer.py:801-832).
 *   prm[B]  : per-view constants; prm[v].bg must point into ONE contiguous device array [B,3]
 *             (prm[v].bg = prm[0].bg + 3 v); P, M, image size, score_flag equal across views;
 *             sh_degree, scale_modifier, cameras may differ per view.
 *   in[B]   : per-view input pointers (any of them may repeat view 0's pointer = shared parameter).
 *   outputs : the views are stacked vertically, each padded to whole tile rows:
 *             out_color [3, Hs, W], out_depth_alpha [2, Hs, W] with Hs from b200gsr_views_geometry
 *             (view v occupies rows [v*Hs/B, v*Hs/B + H)); radii [B,P]; score [B*P] (score_flag).
 *   scratch / saved: sized with the layout queries for (B*P, Hs, W).
 * Backward: dL_dcolor / dL_ddepth_alpha in the same stacked layout; out[B] holds per-view gradient
 * destinations.  out[v].accumulate is a bit mask (1 means3D, 2 opacities, 4 shs/colors, 8 scales,
 * 16 rotations, 32 cov3D): set a bit when that destination is shared with an EARLIER view and the
 * view's contribution must be added instead of written (d_means2D is always per view).
 */
typedef struct b200gsr_view_inputs {
    const float *means3D, *shs, *colors_precomp, *opacities, *scales, *rotations, *cov3D_precomp;
} b200gsr_view_inputs;
typedef struct b200gsr_view_grads {
    float *d_means3D, *d_means2D, *d_shs, *d_colors, *d_opacities, *d_scales, *d_rotations, *d_cov3D;
    uint32_t accumulate;
} b200gsr_view_grads;
int b200gsr_views_geometry(int32_t B, int32_t H, int32_t W, int32_t* stacked_height);
int b200gsr_forward_views(int32_t B, const b200gsr_params* prm, const b200gsr_view_inputs* in,
                          float* out_color, float* out_depth_alpha, int32_t* radii, float* score,
                          void* scratch, size_t scratch_bytes, void* saved, size_t saved_bytes,
                          uint64_t max_pairs, uint32_t flags, uint32_t* host_notify, uint32_t notify_seq,
                          void* stream);
int b200gsr_backward_views(int32_t B, const b200gsr_params* prm, const b200gsr_view_inputs* in,
                           const int32_t* radii, const float* out_depth_alpha, const float* dL_dcolor,
                           const float* dL_ddepth_alpha, void* saved, size_t saved_bytes, uint64_t max_pairs,
                           const b200gsr_view_grads* out, void* stream);

/* Frustum test only (replaces _C.mark_visible; DreamScene never calls it): visible[P] bytes. */
int b200gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix,
                         const float* projmatrix, uint8_t* visible, void* stream);

/*
 * SURVEY.md 8(f2): scene assembly = activations + group concatenation + augmentation noise of
 * scene_render (/root/reference/scene_gaussian.py:753-857; gs_renderer.py:464-488) as one kernel,
 * and its backward as one kernel.  `groups` is a HOST array of `num_groups` (<= B200GSR_MAX_GROUPS)
 * entries holding DEVICE pointers to each group's raw leaf parameters
 *   xyz[n,3] opacity[n,1] scaling[n,3] rotation[n,4] (16-byte aligned) f_dc[n,1,3] f_rest[n,M-1,3]
 * Outputs are the packed rasterizer inputs for P = sum n rows:
 *   means3D[P,3] = xyz, opacities[P,1] = sigmoid, scales[P,3] = exp (+ noise, clamped at 0),
 *   rotations[P,4] = q / max(|q|, 1e-12), shs[P,M,3] = cat(f_dc, f_rest) (+ noise).
 * Noise (reference: v + randn * (0.2**0.5 * v [/ 4 for scales])): shs_noise / scale_noise are the
 * coefficients (0 = off, reference value 0.2**0.5); z_shs[P,M,3] / z_scales[P,3] are standard-normal
 * draws supplied by the caller (same tensors in forward and backward), or NULL to generate them in
 * the kernel from `seed` (counter-based Philox4x32-10; nothing is stored, backward regenerates).
 * Backward: d_* are the gradients w.r.t. the packed outputs, `grads` the per-group destinations
 * (same shapes as the raw parameters, fully overwritten).
 * num_views = B > 1 (the views of one training step, each with its own augmentation): the raw parameters
 * are read once; `scales` is [B,P,3] and `shs` [B,P,M,3] (z_scales [B,P,3], z_shs [B,P,M,3] or Philox
 * streams per view), means3D / opacities / rotations are written once; the backward sums the per-view
 * gradients of scales / shs in registers and writes every leaf gradient once.
 */
#define B200GSR_MAX_GROUPS 24
#define B200GSR_MAX_VIEWS 16
typedef struct b200gsr_group {
    const float *xyz, *opacity, *scaling, *rotation, *f_dc, *f_rest;
    int32_t n;
} b200gsr_group;
typedef struct b200gsr_group_grad {
    float *xyz, *opacity, *scaling, *rotation, *f_dc, *f_rest;
} b200gsr_group_grad;
int b200gsr_assemble_forward(int32_t num_groups, const b200gsr_group* groups, int32_t M, int32_t num_views,
                             float shs_noise, float scale_noise, const float* z_shs, const float* z_scales,
                             uint64_t seed, float* means3D, float* opacities, float* scales, float* rotations,
                             float* shs, void* stream);
int b200gsr_assemble_backward(int32_t num_groups, const b200gsr_group* groups, const b200gsr_group_grad* grads,
                              int32_t M, int32_t num_views, float shs_noise, float scale_noise, const float* z_shs,
                              const float* z_scales, uint64_t seed, const float* d_means3D,
                              const float* d_opacities, const float* d_scales, const float* d_rotations,
                              const float* d_shs, void* stream);

/*
 * SURVEY.md 8(f1, post-processing half): depth/alpha -> normalised disparity of
 * /root/reference/scene_gaussian.py:871-881 for a batch of B views without any host synchronisation.
 *   depth_alpha [B,2,N] (N = H*W; channel 1 = transmittance), focal [B] (device), out_disp [B,N],
 *   stats = 32*B bytes of device scratch that must be kept for the backward.
 * Backward: g_disp [B,N] = dL/d out_disp, g_alpha [B,N] or NULL = dL/d alpha from other consumers of the
 * alpha channel; d_depth_alpha [B,2,N] is fully overwritten.  `stats` is updated in place (pass a copy
 * of the forward's record if the backward may run more than once).
 */
int b200gsr_disparity_forward(int32_t B, int32_t N, const float* depth_alpha, const float* focal,
                              float* out_disp, void* stats, void* stream);
int b200gsr_disparity_backward(int32_t B, int32_t N, const float* depth_alpha, const float* focal,
                               const float* g_disp, const float* g_alpha, void* stats,
                               float* d_depth_alpha, void* stream);

/*
 * SURVEY.md 8(f4): densification / pruning primitives (/root/reference/gs_renderer.py:854-1087).
 * All pointers are device pointers; `scratch` = b200gsr_densify_scratch_bytes(P) bytes.
 *
 * densify_stats  : add_densification_stats + the max_radii2D update for the view just rendered:
 *                  where radii > 0: accum += |viewspace_grad[:, :2]|, denom += 1, max_radii2D = max(., radii)
 * densify_plan   : the per-Gaussian decisions of densify_and_prune (clone / split / prune, in the
 *                  reference's order and with its quirks) + prefix sums.  totals5 (device uint32[5]) =
 *                  {kept originals, surviving clones, surviving split parents, split parents, sum};
 *                  the new point count is totals5[0] + totals5[1] + N * totals5[2].
 *                  dense_extent = percent_dense * extent; big_ws = 0.1 * extent or <= 0 (max_screen_size
 *                  is None); child_div = 0.8 * N as float32.
 * densify_map    : src_map[int32, new count]: bits 0..29 = source row, bits 30..31 = 0 original / 1 clone /
 *                  2 split child, in the reference's output order [originals | clones | children, N blocks];
 *                  child_draw[N * totals5[2]] = row of the reference's torch.normal(std=stds) draw each
 *                  child consumes.
 * compact_plan   : keep mask (uint8) -> src_map of the kept rows and their count (prune_points).
 * gather_rows    : out[p, :] = in[src_map[p], :] for rows of `row_floats` floats; with zero_appended, rows
 *                  whose source is a clone/child become zeros (Adam moments, statistics).
 * split_children : xyz / log-scales of the children (rows >= first_child of the new arrays) from the
 *                  parents' raw parameters and the caller's standard-normal draws z[N * split parents, 3].
 * kth_smallest   : *out = k-th smallest (0-based) of v[n]: the percentile threshold of prune_gaussians
 *                  without a sort.  scratch >= 1032 bytes.
 */
int b200gsr_densify_stats(int32_t P, const float* viewspace_grad, const int32_t* radii, float* accum,
                          float* denom, float* max_radii2D, void* stream);
size_t b200gsr_densify_scratch_bytes(int32_t P);
int b200gsr_densify_plan(int32_t P, const float* accum, const float* denom, const float* scaling,
                         const float* opacity, float max_grad, float dense_extent, float min_opacity,
                         float big_ws, float child_div, void* scratch, uint32_t* totals5, void* stream);
int b200gsr_densify_map(int32_t P, int32_t N, const void* scratch, const uint32_t* totals5,
                        int32_t* src_map, int32_t* child_draw, void* stream);
int b200gsr_compact_plan(int32_t P, const uint8_t* keep, void* scratch, int32_t* src_map, uint32_t* count,
                         void* stream);
int b200gsr_gather_rows(int32_t n_out, int32_t row_floats, const int32_t* src_map, const float* in, float* out,
                        int32_t zero_appended, void* stream);
int b200gsr_split_children(int32_t n_out, int32_t first_child, float child_div, const int32_t* src_map,
                           const int32_t* child_draw, const float* xyz, const float* scaling,
                           const float* rotation, const float* z, float* xyz_out, float* scaling_out,
                           void* stream);
int b200gsr_kth_smallest(int32_t n, const float* v, uint32_t k, void* scratch, float* out, void* stream);

/*
 * SURVEY.md 8(f3): replaces simple_knn._C.distCUDA2 (un-vendored; /root/reference/gs_renderer.py:9,590-593):
 * out[i] = mean of the squared distances from points[i] to its 3 nearest OTHER points (points f32[P,3]).
 * `scratch` = b200gsr_dist2_scratch_bytes(P) bytes of device memory.
 */
size_t b200gsr_dist2_scratch_bytes(int32_t P);
int b200gsr_dist2_knn3(int32_t P, const float* points, float* out, void* scratch, size_t scratch_bytes,
                       void* stream);

/*
 * Optional per-stage device timing for benchmarks (no upstream equivalent).  Process-wide and not
 * thread-safe.  enable(max_calls>0) allocates CUDA events; every later forward/backward call
 * (up to max_calls each) records events around its stages on the call's stream; read() waits for
 * that call and returns elapsed milliseconds:
 *   forward  ms[5] = {project_sh, scan_order, scatter, tile_sort(2 kernels), composite_fwd}
 *   backward ms[2] = {composite_bwd, project_bwd}
 * enable(0) frees everything.
 */
int b200gsr_profile_enable(int32_t max_calls);
/*
 * Diagnostics (no upstream equivalent; process-wide, not thread-safe): while `device_counters`
 * (16 zero-initialised uint64 in device memory) is set, the composite kernels run in their
 * instrumented instantiation and accumulate
 *   [0] (warp, Gaussian) pairs evaluated by the backward  [1] ... with >= 1 contributing pixel
 *   [2] contributing (pixel, Gaussian) pairs              [3..8] histogram of contributing lanes per
 *   pair: 1, 2, 3-4, 5-8, 9-16, 17-32                     [10] pairs evaluated by the forward
 *   [11] blended (pixel, Gaussian) pairs in the forward.
 *   [16..20] forward load balance (globaltimer ns): sum of CTA busy time, last exit, ~(first entry), CTAs,
 *   longest tile;  [21..26] the same for the backward's warps + most evaluations / longest time of one item.
 * The buffer holds 32 zeroed uint64.
 * bench.py uses them (outside the timed region) for the pair-evaluation roofline.  NULL switches back.
 */
int b200gsr_debug_counters(unsigned long long* device_counters);
int b200gsr_profile_counts(int32_t* n_forward, int32_t* n_backward);
int b200gsr_profile_read(int32_t is_backward, int32_t call, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* B200GSR_H */
