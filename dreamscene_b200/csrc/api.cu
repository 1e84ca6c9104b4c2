// C ABI (include/b200gsr.h): argument validation, buffer layouts, launch sequencing.
#include "common.cuh"

#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <mutex>

#ifndef B200GSR_NO_NVTX
#include <nvtx3/nvToolsExt.h>   // header-only; a no-op unless a profiler is attached
#define GSR_RANGE_PUSH(name) nvtxRangePushA(name)
#define GSR_RANGE_POP() nvtxRangePop()
#else
#define GSR_RANGE_PUSH(name) ((void)0)
#define GSR_RANGE_POP() ((void)0)
#endif

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

int check_cuda(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return B200GSR_OK;
    return fail(B200GSR_ERR_CUDA, "%s: %s", what, cudaGetErrorString(e));
}

// ---- optional per-stage timing (process-wide, not thread-safe; used by bench.py only) ----------
enum { kFwdEvents = 6, kBwdEvents = 3 };
struct Prof {
    int max_calls = 0;
    int nfwd = 0, nbwd = 0;
    cudaEvent_t* fwd = nullptr;   // [max_calls][kFwdEvents]
    cudaEvent_t* bwd = nullptr;   // [max_calls][kBwdEvents]
} g_prof;

void prof_mark_fwd(int k, cudaStream_t s) {
    if (g_prof.max_calls > 0 && g_prof.nfwd < g_prof.max_calls)
        cudaEventRecord(g_prof.fwd[g_prof.nfwd * kFwdEvents + k], s);
}
void prof_mark_bwd(int k, cudaStream_t s) {
    if (g_prof.max_calls > 0 && g_prof.nbwd < g_prof.max_calls)
        cudaEventRecord(g_prof.bwd[g_prof.nbwd * kBwdEvents + k], s);
}

// ---- per-device state, created lazily under a mutex and never destroyed: SM count + a forked
// stream that lets the two tile-sort size classes run concurrently.
struct DeviceState {
    bool ready = false;
    int num_sms = 148;
    cudaStream_t stream = nullptr;
    cudaEvent_t fork = nullptr, join = nullptr;
};
DeviceState g_dev[64];
unsigned long long* g_stats = nullptr;   // b200gsr_debug_counters (process-wide, diagnostics only)
std::mutex g_dev_mutex;

// Returns nullptr only if the device ordinal is out of range or CUDA itself fails.
DeviceState* device_state() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    DeviceState& s = g_dev[dev];
    if (s.ready) return &s;                       // written once under the mutex
    std::lock_guard<std::mutex> lock(g_dev_mutex);
    if (s.ready) return &s;
    int nsm = 148;
    if (cudaDeviceGetAttribute(&nsm, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && nsm > 0) s.num_sms = nsm;
    // the side stream is optional: without it the two sort kernels simply run back to back
    cudaStream_t st = nullptr;
    cudaEvent_t ef = nullptr, ej = nullptr;
    if (cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking) == cudaSuccess &&
        cudaEventCreateWithFlags(&ef, cudaEventDisableTiming) == cudaSuccess &&
        cudaEventCreateWithFlags(&ej, cudaEventDisableTiming) == cudaSuccess) {
        s.stream = st; s.fork = ef; s.join = ej;
    } else {
        if (ef) cudaEventDestroy(ef);
        if (ej) cudaEventDestroy(ej);
        if (st) cudaStreamDestroy(st);
        cudaGetLastError();   // clear the non-sticky creation error
    }
    s.ready = true;
    return &s;
}

int validate_inputs(const b200gsr_params* p, const float* means3D, const float* shs,
                    const float* colors, const float* opac, const float* scales,
                    const float* rots, const float* cov3d) {
    if (!p) return fail(B200GSR_ERR_BAD_ARG, "params is null");
    if (p->P < 0 || p->image_height < 0 || p->image_width < 0)
        return fail(B200GSR_ERR_BAD_ARG, "negative size");
    if (p->image_height > 65535 * 16 || p->image_width > 65535 * 16)
        return fail(B200GSR_ERR_UNSUPPORTED, "image larger than 65535 tiles per axis");
    if (!p->bg || !p->viewmatrix || !p->projmatrix || !p->campos)
        return fail(B200GSR_ERR_BAD_ARG, "bg/viewmatrix/projmatrix/campos must be device pointers");
    if (p->P > 0) {
        if (!means3D || !opac) return fail(B200GSR_ERR_BAD_ARG, "means3D/opacities are required");
        if ((shs != nullptr) == (colors != nullptr))
            return fail(B200GSR_ERR_BAD_ARG, "Please provide excatly one of either SHs or precomputed colors!");
        const bool has_sr = scales != nullptr || rots != nullptr;
        if (((scales == nullptr || rots == nullptr) && cov3d == nullptr) || (has_sr && cov3d != nullptr))
            return fail(B200GSR_ERR_BAD_ARG,
                        "Please provide exactly one of either scale/rotation pair or precomputed 3D covariance!");
        if (shs) {
            if (p->sh_degree < 0 || p->sh_degree > 3)
                return fail(B200GSR_ERR_UNSUPPORTED, "sh_degree %d not in 0..3", p->sh_degree);
            if (p->M < (p->sh_degree + 1) * (p->sh_degree + 1) || p->M > 16)
                return fail(B200GSR_ERR_BAD_ARG, "M=%d inconsistent with sh_degree=%d (need (deg+1)^2 <= M <= 16)",
                            p->M, p->sh_degree);
        }
    }
    return B200GSR_OK;
}

}  // namespace

extern "C" {

int b200gsr_version(void) { return B200GSR_VERSION; }

const char* b200gsr_last_error(void) { return g_err; }

int b200gsr_saved_layout_query(int32_t P, int32_t H, int32_t W, uint64_t max_pairs,
                               int32_t with_backward, b200gsr_saved_layout* out) {
    if (!out || P < 0 || H < 0 || W < 0) return fail(B200GSR_ERR_BAD_ARG, "bad layout query");
    if (max_pairs > 0xfffffff0ull) return fail(B200GSR_ERR_UNSUPPORTED, "max_pairs must fit in 32 bits");
    const GsrTileGrid g = gsr_grid(H, W);
    size_t off = 0;
    out->header = off;      off = align_up(off + GSR_H_WORDS * sizeof(uint32_t));
    out->tile_start = off;  off = align_up(off + ((size_t)g.ntiles + 1) * sizeof(uint32_t));
    out->work_order = off;  off = align_up(off + (size_t)g.ntiles * sizeof(uint32_t));
    out->n_contrib = off;   off = align_up(off + (size_t)H * W * sizeof(uint32_t));
    out->keys = off;        off = align_up(off + ((size_t)max_pairs + 2) * sizeof(uint64_t));
    out->geom = off;        off = align_up(off + (size_t)P * sizeof(GsrRec));
    out->dgeom = off;       off = align_up(off + (with_backward ? (size_t)P * 12 * sizeof(float) : 0));
    out->bwd_items = off;   off = align_up(off + (with_backward ? (size_t)GSR_BWD_CLASSES * g.ntiles * 8 * sizeof(uint32_t) : 0));
    out->total = off;
    return B200GSR_OK;
}

int b200gsr_scratch_layout_query(int32_t P, int32_t H, int32_t W, uint64_t max_pairs,
                                 b200gsr_scratch_layout* out) {
    if (!out || P < 0 || H < 0 || W < 0) return fail(B200GSR_ERR_BAD_ARG, "bad layout query");
    if (max_pairs > 0xfffffff0ull) return fail(B200GSR_ERR_UNSUPPORTED, "max_pairs must fit in 32 bits");
    const GsrTileGrid g = gsr_grid(H, W);
    size_t off = 0;
    out->counters = off;    off = align_up(off + GSR_NCOUNTERS * sizeof(uint32_t));
    out->tile_count = off;  off = align_up(off + (size_t)GSR_COPIES * g.ntiles * sizeof(uint32_t));
    out->tile_cursor = off; off = align_up(off + (size_t)GSR_COPIES * g.ntiles * sizeof(uint32_t));
    out->rectdepth = off;   off = align_up(off + (size_t)P * sizeof(uint4));
    {
        const size_t nblk = (size_t)gsr_ms_blocks(P);
        out->ms_hist = off; off = align_up(off + (gsr_use_multisplit(g.ntiles) ? nblk * g.ntiles * sizeof(uint32_t) : 0));
    }
    out->total = off;
    return B200GSR_OK;
}

int b200gsr_forward(const b200gsr_params* prm, const float* means3D, const float* shs,
                    const float* colors_precomp, const float* opacities, const float* scales,
                    const float* rotations, const float* cov3D_precomp, float* out_color,
                    float* out_depth_alpha, int32_t* radii, float* score, void* scratch,
                    size_t scratch_bytes, void* saved, size_t saved_bytes, uint64_t max_pairs,
                    uint32_t flags, uint32_t* host_notify, uint32_t notify_seq, void* stream) {
    int rc = validate_inputs(prm, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp);
    if (rc) return rc;
    if (!out_color || !out_depth_alpha || (prm->P > 0 && !radii) || !scratch || !saved)
        return fail(B200GSR_ERR_BAD_ARG, "null output/workspace pointer");
    if (prm->score_flag && prm->P > 0 && !score)
        return fail(B200GSR_ERR_BAD_ARG, "score_flag set but score buffer is null");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    GsrFwdArgs a;
    a.prm = *prm;
    const int with_bwd = (flags & B200GSR_FWD_NO_BACKWARD) ? 0 : 1;
    if ((rc = b200gsr_scratch_layout_query(prm->P, prm->image_height, prm->image_width, max_pairs, &a.sl))) return rc;
    if ((rc = b200gsr_saved_layout_query(prm->P, prm->image_height, prm->image_width, max_pairs, with_bwd, &a.vl))) return rc;
    if (scratch_bytes < a.sl.total || saved_bytes < a.vl.total)
        return fail(B200GSR_ERR_WORKSPACE, "workspace too small: scratch %zu < %zu or saved %zu < %zu",
                    scratch_bytes, a.sl.total, saved_bytes, a.vl.total);
    a.means3D = means3D; a.shs = shs; a.colors = colors_precomp; a.opac = opacities;
    a.scales = scales; a.rots = rotations; a.cov3d = cov3D_precomp;
    a.out_color = out_color; a.out_depth_alpha = out_depth_alpha; a.score = score; a.radii = radii;
    a.scratch = static_cast<uint8_t*>(scratch); a.saved = static_cast<uint8_t*>(saved);
    a.max_pairs = (uint32_t)max_pairs;
    a.host_notify = host_notify; a.notify_seq = notify_seq;
    a.flags = flags; a.num_sms = ds->num_sms; a.stats = g_stats;
    a.view = 0; a.num_views = 1; a.P_view = prm->P; a.gy_view = gsr_grid(prm->image_height, prm->image_width).gy;
    a.stream = static_cast<cudaStream_t>(stream);

    // The queue counters and the per-tile pair counters (contiguous at the start of scratch) must be
    // zero before the count kernel runs.  On the main path (smem multisplit binning, P > 0) the
    // project_sh prologue zeroes them; only the large-grid fallback (project_sh itself counts with
    // global atomics) and the P == 0 case need a memset node.
    {
        const GsrTileGrid tg = gsr_grid(prm->image_height, prm->image_width);
        if (!gsr_use_multisplit(tg.ntiles) || prm->P == 0) {
            const size_t nbytes = gsr_use_multisplit(tg.ntiles) ? a.sl.tile_count + (size_t)tg.ntiles * sizeof(uint32_t)
                                                                : a.sl.tile_cursor;
            if ((rc = check_cuda(cudaMemsetAsync(a.scratch, 0, nbytes, a.stream), "memset"))) return rc;
        }
    }
    prof_mark_fwd(0, a.stream);
    GSR_RANGE_PUSH("b200gsr.project_sh+count");
    rc = check_cuda(gsr_launch_project(a), "project_sh");
    if (!rc) rc = check_cuda(gsr_launch_count(a), "tile_count");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_fwd(1, a.stream);
    GSR_RANGE_PUSH("b200gsr.scan_order");
    rc = check_cuda(gsr_launch_scan(a), "scan_order");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_fwd(2, a.stream);
    GSR_RANGE_PUSH("b200gsr.scatter");
    rc = check_cuda(gsr_launch_scatter(a), "scatter");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_fwd(3, a.stream);
    GSR_RANGE_PUSH("b200gsr.tile_sort");
    rc = check_cuda(gsr_launch_sort(a, ds->stream, ds->fork, ds->join), "tile_sort");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_fwd(4, a.stream);
    GSR_RANGE_PUSH("b200gsr.composite_fwd");
    rc = check_cuda(gsr_launch_composite_fwd(a), "composite_fwd");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_fwd(5, a.stream);
    if (g_prof.max_calls > 0 && g_prof.nfwd < g_prof.max_calls) ++g_prof.nfwd;
    return B200GSR_OK;
}

int b200gsr_backward_ex(const b200gsr_params* prm, const float* means3D, const float* shs,
                     const float* colors_precomp, const float* opacities, const float* scales,
                     const float* rotations, const float* cov3D_precomp, const int32_t* radii,
                     const float* out_depth_alpha, const float* dL_dcolor,
                     const float* dL_ddepth_alpha, void* saved, size_t saved_bytes,
                     void* /*scratch*/, size_t /*scratch_bytes*/, uint64_t max_pairs, float* d_means3D,
                     float* d_means2D, float* d_shs, float* d_colors, float* d_opacities,
                     float* d_scales, float* d_rotations, float* d_cov3D, int32_t dsh_coefs, void* stream) {
    int rc = validate_inputs(prm, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp);
    if (rc) return rc;
    if (prm->P == 0) return B200GSR_OK;
    if (shs && dsh_coefs != 0 && dsh_coefs != -1 &&
        (dsh_coefs < (prm->sh_degree + 1) * (prm->sh_degree + 1) || dsh_coefs > prm->M))
        return fail(B200GSR_ERR_BAD_ARG, "dsh_coefs=%d must be 0, -1 or in [(sh_degree+1)^2, M]", dsh_coefs);
    if (!shs && dsh_coefs < 0) return fail(B200GSR_ERR_BAD_ARG, "dsh_coefs=-1 (factored SH gradient) needs shs");
    if (!radii || !out_depth_alpha || !dL_dcolor || !dL_ddepth_alpha || !saved)
        return fail(B200GSR_ERR_BAD_ARG, "null saved-state/gradient pointer");
    if (!d_means3D || !d_means2D || !d_opacities || (shs && !d_shs) || (colors_precomp && !d_colors) ||
        (cov3D_precomp && !d_cov3D) || (!cov3D_precomp && (!d_scales || !d_rotations)))
        return fail(B200GSR_ERR_BAD_ARG, "null gradient output pointer");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    GsrBwdArgs a;
    a.prm = *prm;
    a.sl = b200gsr_scratch_layout{};
    if ((rc = b200gsr_saved_layout_query(prm->P, prm->image_height, prm->image_width, max_pairs, 1, &a.vl))) return rc;
    if (saved_bytes < a.vl.total)
        return fail(B200GSR_ERR_WORKSPACE, "saved buffer too small for backward: %zu < %zu (was the forward "
                    "run with B200GSR_FWD_NO_BACKWARD?)", saved_bytes, a.vl.total);
    a.means3D = means3D; a.shs = shs; a.colors = colors_precomp; a.opac = opacities;
    a.scales = scales; a.rots = rotations; a.cov3d = cov3D_precomp;
    a.radii = radii; a.out_depth_alpha = out_depth_alpha;
    a.dL_dcolor = dL_dcolor; a.dL_ddepth_alpha = dL_ddepth_alpha;
    a.saved = static_cast<uint8_t*>(saved); a.scratch = nullptr;
    a.max_pairs = (uint32_t)max_pairs;
    a.d_means3D = d_means3D; a.d_means2D = d_means2D; a.d_shs = d_shs; a.d_colors = d_colors;
    a.d_opac = d_opacities; a.d_scales = d_scales; a.d_rots = d_rotations; a.d_cov3d = d_cov3D;
    a.num_sms = ds->num_sms; a.stats = g_stats;
    a.dsh_coefs = dsh_coefs;
    a.view = 0; a.num_views = 1; a.P_view = prm->P; a.gy_view = gsr_grid(prm->image_height, prm->image_width).gy;
    a.accumulate = 0;
    a.stream = static_cast<cudaStream_t>(stream);

    // no memsets: the work-queue counters and the gradient accumulators live in `saved`, zeroed by
    // the forward and restored to zero by project_bwd
    prof_mark_bwd(0, a.stream);
    GSR_RANGE_PUSH("b200gsr.composite_bwd");
    rc = check_cuda(gsr_launch_composite_bwd(a), "composite_bwd");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_bwd(1, a.stream);
    GSR_RANGE_PUSH("b200gsr.project_bwd");
    rc = check_cuda(gsr_launch_project_bwd(a), "project_bwd");
    GSR_RANGE_POP();
    if (rc) return rc;
    prof_mark_bwd(2, a.stream);
    if (g_prof.max_calls > 0 && g_prof.nbwd < g_prof.max_calls) ++g_prof.nbwd;
    return B200GSR_OK;
}

int b200gsr_backward(const b200gsr_params* prm, const float* means3D, const float* shs,
                     const float* colors_precomp, const float* opacities, const float* scales,
                     const float* rotations, const float* cov3D_precomp, const int32_t* radii,
                     const float* out_depth_alpha, const float* dL_dcolor,
                     const float* dL_ddepth_alpha, void* saved, size_t saved_bytes,
                     void* scratch, size_t scratch_bytes, uint64_t max_pairs, float* d_means3D,
                     float* d_means2D, float* d_shs, float* d_colors, float* d_opacities,
                     float* d_scales, float* d_rotations, float* d_cov3D, void* stream) {
    return b200gsr_backward_ex(prm, means3D, shs, colors_precomp, opacities, scales, rotations, cov3D_precomp, radii,
                               out_depth_alpha, dL_dcolor, dL_ddepth_alpha, saved, saved_bytes, scratch, scratch_bytes,
                               max_pairs, d_means3D, d_means2D, d_shs, d_colors, d_opacities, d_scales, d_rotations,
                               d_cov3D, 0, stream);
}

// ---------------------------------------------------------------------------------------------
// Multi-view entry points (SURVEY.md 8 f1): B views of the same image size in ONE binning / sort /
// composite pass.  The views are stacked vertically into an image of B * gy tile rows and view v's
// Gaussians become the virtual Gaussians [v*P, (v+1)*P): only the two per-Gaussian stages run per view
// (each with its own camera and, if the caller wishes, its own parameter tensors).
// ---------------------------------------------------------------------------------------------
static int check_views(int32_t B, const b200gsr_params* prm, const b200gsr_view_inputs* in) {
    if (B < 1 || B > B200GSR_MAX_VIEWS) return fail(B200GSR_ERR_UNSUPPORTED, "number of views %d not in 1..%d", B, B200GSR_MAX_VIEWS);
    if (!prm || !in) return fail(B200GSR_ERR_BAD_ARG, "null view array");
    for (int v = 0; v < B; ++v) {
        int rc = validate_inputs(&prm[v], in[v].means3D, in[v].shs, in[v].colors_precomp, in[v].opacities, in[v].scales,
                                 in[v].rotations, in[v].cov3D_precomp);
        if (rc) return rc;
        if (prm[v].P != prm[0].P || prm[v].M != prm[0].M || prm[v].image_height != prm[0].image_height ||
            prm[v].image_width != prm[0].image_width || prm[v].score_flag != prm[0].score_flag)
            return fail(B200GSR_ERR_BAD_ARG, "view %d: P, M, image size and score_flag must equal view 0's", v);
        if (prm[v].bg != prm[0].bg + 3 * v)
            return fail(B200GSR_ERR_BAD_ARG, "view %d: backgrounds must be one contiguous device array [B,3] (prm[v].bg = prm[0].bg + 3 v)", v);
        if ((in[v].shs != nullptr) != (in[0].shs != nullptr) || (in[v].cov3D_precomp != nullptr) != (in[0].cov3D_precomp != nullptr))
            return fail(B200GSR_ERR_BAD_ARG, "view %d: all views must use the same input kinds", v);
    }
    if ((long long)B * prm[0].P > 0x3fffffffLL) return fail(B200GSR_ERR_UNSUPPORTED, "B * P too large");
    return B200GSR_OK;
}

int b200gsr_views_geometry(int32_t B, int32_t H, int32_t W, int32_t* stacked_height) {
    if (B < 1 || H < 0 || W < 0 || !stacked_height) return fail(B200GSR_ERR_BAD_ARG, "bad views_geometry arguments");
    *stacked_height = B * gsr_grid(H, W).gy * GSR_TILE;
    return B200GSR_OK;
}

int b200gsr_forward_views(int32_t B, const b200gsr_params* prm, const b200gsr_view_inputs* in, float* out_color,
                          float* out_depth_alpha, int32_t* radii, float* score, void* scratch, size_t scratch_bytes,
                          void* saved, size_t saved_bytes, uint64_t max_pairs, uint32_t flags, uint32_t* host_notify,
                          uint32_t notify_seq, void* stream) {
    int rc = check_views(B, prm, in);
    if (rc) return rc;
    const int P = prm[0].P, H = prm[0].image_height, W = prm[0].image_width;
    if (!out_color || !out_depth_alpha || (P > 0 && !radii) || !scratch || !saved)
        return fail(B200GSR_ERR_BAD_ARG, "null output/workspace pointer");
    if (prm[0].score_flag && P > 0 && !score) return fail(B200GSR_ERR_BAD_ARG, "score_flag set but score buffer is null");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    const GsrTileGrid g1 = gsr_grid(H, W);
    const int Hs = B * g1.gy * GSR_TILE;
    GsrFwdArgs a;
    const int with_bwd = (flags & B200GSR_FWD_NO_BACKWARD) ? 0 : 1;
    if ((rc = b200gsr_scratch_layout_query(B * P, Hs, W, max_pairs, &a.sl))) return rc;
    if ((rc = b200gsr_saved_layout_query(B * P, Hs, W, max_pairs, with_bwd, &a.vl))) return rc;
    if (scratch_bytes < a.sl.total || saved_bytes < a.vl.total)
        return fail(B200GSR_ERR_WORKSPACE, "workspace too small: scratch %zu < %zu or saved %zu < %zu",
                    scratch_bytes, a.sl.total, saved_bytes, a.vl.total);
    a.out_color = out_color; a.out_depth_alpha = out_depth_alpha; a.score = score; a.radii = radii;
    a.scratch = static_cast<uint8_t*>(scratch); a.saved = static_cast<uint8_t*>(saved);
    a.max_pairs = (uint32_t)max_pairs;
    a.host_notify = host_notify; a.notify_seq = notify_seq;
    a.flags = flags; a.num_sms = ds->num_sms; a.stats = g_stats;
    a.num_views = B; a.P_view = P; a.gy_view = g1.gy;
    a.stream = static_cast<cudaStream_t>(stream);
    const int ntiles = g1.gx * g1.gy * B;
    if (!gsr_use_multisplit(ntiles) || P == 0) {
        const size_t nbytes = gsr_use_multisplit(ntiles) ? a.sl.tile_count + (size_t)ntiles * sizeof(uint32_t) : a.sl.tile_cursor;
        if ((rc = check_cuda(cudaMemsetAsync(a.scratch, 0, nbytes, a.stream), "memset"))) return rc;
    }
    GSR_RANGE_PUSH("b200gsr.views.project_sh");
    for (int v = 0; v < B && !rc; ++v) {
        a.prm = prm[v]; a.view = v;
        a.means3D = in[v].means3D; a.shs = in[v].shs; a.colors = in[v].colors_precomp; a.opac = in[v].opacities;
        a.scales = in[v].scales; a.rots = in[v].rotations; a.cov3d = in[v].cov3D_precomp;
        rc = check_cuda(gsr_launch_project(a), "project_sh");
    }
    GSR_RANGE_POP();
    if (rc) return rc;
    a.prm = prm[0]; a.view = 0;     // per-view constants are not used past this point (bg is indexed by tile row)
    GSR_RANGE_PUSH("b200gsr.views.binning+sort+composite");
    rc = check_cuda(gsr_launch_count(a), "tile_count");
    if (!rc) rc = check_cuda(gsr_launch_scan(a), "scan_order");
    if (!rc) rc = check_cuda(gsr_launch_scatter(a), "scatter");
    if (!rc) rc = check_cuda(gsr_launch_sort(a, ds->stream, ds->fork, ds->join), "tile_sort");
    if (!rc) rc = check_cuda(gsr_launch_composite_fwd(a), "composite_fwd");
    GSR_RANGE_POP();
    return rc;
}

int b200gsr_backward_views(int32_t B, const b200gsr_params* prm, const b200gsr_view_inputs* in, const int32_t* radii,
                           const float* out_depth_alpha, const float* dL_dcolor, const float* dL_ddepth_alpha,
                           void* saved, size_t saved_bytes, uint64_t max_pairs, const b200gsr_view_grads* out,
                           void* stream) {
    int rc = check_views(B, prm, in);
    if (rc) return rc;
    const int P = prm[0].P, H = prm[0].image_height, W = prm[0].image_width;
    if (P == 0) return B200GSR_OK;
    if (!radii || !out_depth_alpha || !dL_dcolor || !dL_ddepth_alpha || !saved || !out)
        return fail(B200GSR_ERR_BAD_ARG, "null saved-state/gradient pointer");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    const GsrTileGrid g1 = gsr_grid(H, W);
    const int Hs = B * g1.gy * GSR_TILE;
    GsrBwdArgs a;
    a.sl = b200gsr_scratch_layout{};
    if ((rc = b200gsr_saved_layout_query(B * P, Hs, W, max_pairs, 1, &a.vl))) return rc;
    if (saved_bytes < a.vl.total) return fail(B200GSR_ERR_WORKSPACE, "saved buffer too small for backward: %zu < %zu", saved_bytes, a.vl.total);
    a.radii = radii; a.out_depth_alpha = out_depth_alpha; a.dL_dcolor = dL_dcolor; a.dL_ddepth_alpha = dL_ddepth_alpha;
    a.saved = static_cast<uint8_t*>(saved); a.scratch = nullptr; a.max_pairs = (uint32_t)max_pairs;
    a.num_sms = ds->num_sms; a.stats = g_stats;
    a.num_views = B; a.P_view = P; a.gy_view = g1.gy; a.dsh_coefs = 0;
    a.stream = static_cast<cudaStream_t>(stream);
    a.prm = prm[0]; a.view = 0; a.accumulate = 0;
    a.means3D = in[0].means3D; a.shs = in[0].shs; a.colors = in[0].colors_precomp; a.opac = in[0].opacities;
    a.scales = in[0].scales; a.rots = in[0].rotations; a.cov3d = in[0].cov3D_precomp;
    GSR_RANGE_PUSH("b200gsr.views.composite_bwd");
    rc = check_cuda(gsr_launch_composite_bwd(a), "composite_bwd");
    GSR_RANGE_POP();
    if (rc) return rc;
    GSR_RANGE_PUSH("b200gsr.views.project_bwd");
    for (int v = 0; v < B && !rc; ++v) {
        const b200gsr_view_grads& o = out[v];
        if (!o.d_means3D || !o.d_means2D || !o.d_opacities || (in[v].shs && !o.d_shs) || (in[v].colors_precomp && !o.d_colors) ||
            (in[v].cov3D_precomp && !o.d_cov3D) || (!in[v].cov3D_precomp && (!o.d_scales || !o.d_rotations))) {
            rc = fail(B200GSR_ERR_BAD_ARG, "view %d: null gradient output pointer", v);
            break;
        }
        a.prm = prm[v]; a.view = v; a.accumulate = (int)o.accumulate;
        a.means3D = in[v].means3D; a.shs = in[v].shs; a.colors = in[v].colors_precomp; a.opac = in[v].opacities;
        a.scales = in[v].scales; a.rots = in[v].rotations; a.cov3d = in[v].cov3D_precomp;
        a.d_means3D = o.d_means3D; a.d_means2D = o.d_means2D; a.d_shs = o.d_shs; a.d_colors = o.d_colors;
        a.d_opac = o.d_opacities; a.d_scales = o.d_scales; a.d_rots = o.d_rotations; a.d_cov3d = o.d_cov3D;
        rc = check_cuda(gsr_launch_project_bwd(a), "project_bwd");
    }
    GSR_RANGE_POP();
    return rc;
}

int b200gsr_profile_enable(int32_t max_calls) {
    for (int i = 0; i < g_prof.max_calls * kFwdEvents; ++i) cudaEventDestroy(g_prof.fwd[i]);
    for (int i = 0; i < g_prof.max_calls * kBwdEvents; ++i) cudaEventDestroy(g_prof.bwd[i]);
    delete[] g_prof.fwd; delete[] g_prof.bwd;
    g_prof = Prof();
    if (max_calls <= 0) return B200GSR_OK;
    g_prof.fwd = new cudaEvent_t[(size_t)max_calls * kFwdEvents];
    g_prof.bwd = new cudaEvent_t[(size_t)max_calls * kBwdEvents];
    for (int i = 0; i < max_calls * kFwdEvents; ++i)
        if (cudaEventCreate(&g_prof.fwd[i]) != cudaSuccess) return fail(B200GSR_ERR_CUDA, "cudaEventCreate");
    for (int i = 0; i < max_calls * kBwdEvents; ++i)
        if (cudaEventCreate(&g_prof.bwd[i]) != cudaSuccess) return fail(B200GSR_ERR_CUDA, "cudaEventCreate");
    g_prof.max_calls = max_calls;
    return B200GSR_OK;
}

int b200gsr_profile_counts(int32_t* n_forward, int32_t* n_backward) {
    if (n_forward) *n_forward = g_prof.nfwd;
    if (n_backward) *n_backward = g_prof.nbwd;
    return B200GSR_OK;
}

int b200gsr_profile_read(int32_t is_backward, int32_t call, float* ms) {
    if (!ms) return fail(B200GSR_ERR_BAD_ARG, "ms is null");
    const int n = is_backward ? g_prof.nbwd : g_prof.nfwd;
    if (call < 0 || call >= n) return fail(B200GSR_ERR_BAD_ARG, "profile call index %d out of range (%d)", call, n);
    const int ne = is_backward ? kBwdEvents : kFwdEvents;
    cudaEvent_t* ev = (is_backward ? g_prof.bwd : g_prof.fwd) + (size_t)call * ne;
    cudaError_t e = cudaEventSynchronize(ev[ne - 1]);
    if (e != cudaSuccess) return check_cuda(e, "cudaEventSynchronize");
    for (int k = 0; k + 1 < ne; ++k)
        if ((e = cudaEventElapsedTime(&ms[k], ev[k], ev[k + 1])) != cudaSuccess)
            return check_cuda(e, "cudaEventElapsedTime");
    return B200GSR_OK;
}

static int check_groups(int32_t num_groups, const b200gsr_group* groups, int32_t M) {
    if (num_groups < 0 || num_groups > B200GSR_MAX_GROUPS) return fail(B200GSR_ERR_UNSUPPORTED, "num_groups %d not in 0..%d", num_groups, B200GSR_MAX_GROUPS);
    if (num_groups > 0 && !groups) return fail(B200GSR_ERR_BAD_ARG, "groups is null");
    if (M < 1 || M > 16) return fail(B200GSR_ERR_BAD_ARG, "M=%d not in 1..16", M);
    long long total = 0;
    for (int g = 0; g < num_groups; ++g) {
        const b200gsr_group& gr = groups[g];
        if (gr.n < 0) return fail(B200GSR_ERR_BAD_ARG, "group %d: negative size", g);
        if (gr.n > 0 && (!gr.xyz || !gr.opacity || !gr.scaling || !gr.rotation || !gr.f_dc || (M > 1 && !gr.f_rest)))
            return fail(B200GSR_ERR_BAD_ARG, "group %d: null parameter pointer", g);
        if (gr.n > 0 && (reinterpret_cast<uintptr_t>(gr.rotation) & 15u))
            return fail(B200GSR_ERR_BAD_ARG, "group %d: rotation must be 16-byte aligned", g);
        total += gr.n;
    }
    if (total > 0x7fffffffLL) return fail(B200GSR_ERR_UNSUPPORTED, "more than 2^31-1 Gaussians");
    return B200GSR_OK;
}

int b200gsr_assemble_forward(int32_t num_groups, const b200gsr_group* groups, int32_t M, int32_t num_views, float shs_noise,
                             float scale_noise, const float* z_shs, const float* z_scales, uint64_t seed,
                             float* means3D, float* opacities, float* scales, float* rotations, float* shs,
                             void* stream) {
    int rc = check_groups(num_groups, groups, M);
    if (rc) return rc;
    if (!means3D || !opacities || !scales || !rotations || !shs) return fail(B200GSR_ERR_BAD_ARG, "null output pointer");
    if (num_views < 1 || num_views > B200GSR_MAX_VIEWS) return fail(B200GSR_ERR_BAD_ARG, "num_views %d not in 1..%d", num_views, B200GSR_MAX_VIEWS);
    GSR_RANGE_PUSH("b200gsr.assemble_fwd");
    rc = check_cuda(gsr_launch_assemble(false, num_groups, groups, nullptr, M, num_views, shs_noise, scale_noise, z_shs, z_scales,
                                        seed, means3D, opacities, scales, rotations, shs,
                                        static_cast<cudaStream_t>(stream)), "assemble_forward");
    GSR_RANGE_POP();
    return rc;
}

int b200gsr_assemble_backward(int32_t num_groups, const b200gsr_group* groups, const b200gsr_group_grad* grads,
                              int32_t M, int32_t num_views, float shs_noise, float scale_noise, const float* z_shs,
                              const float* z_scales, uint64_t seed, const float* d_means3D,
                              const float* d_opacities, const float* d_scales, const float* d_rotations,
                              const float* d_shs, void* stream) {
    int rc = check_groups(num_groups, groups, M);
    if (rc) return rc;
    if (num_groups > 0 && !grads) return fail(B200GSR_ERR_BAD_ARG, "grads is null");
    for (int g = 0; g < num_groups; ++g)
        if (groups[g].n > 0 && (!grads[g].xyz || !grads[g].opacity || !grads[g].scaling || !grads[g].rotation ||
                                !grads[g].f_dc || (M > 1 && !grads[g].f_rest)))
            return fail(B200GSR_ERR_BAD_ARG, "group %d: null gradient pointer", g);
    if (!d_means3D || !d_opacities || !d_scales || !d_rotations || !d_shs) return fail(B200GSR_ERR_BAD_ARG, "null gradient input");
    if (num_views < 1 || num_views > B200GSR_MAX_VIEWS) return fail(B200GSR_ERR_BAD_ARG, "num_views %d not in 1..%d", num_views, B200GSR_MAX_VIEWS);
    GSR_RANGE_PUSH("b200gsr.assemble_bwd");
    rc = check_cuda(gsr_launch_assemble(true, num_groups, groups, grads, M, num_views, shs_noise, scale_noise, z_shs, z_scales, seed,
                                        const_cast<float*>(d_means3D), const_cast<float*>(d_opacities),
                                        const_cast<float*>(d_scales), const_cast<float*>(d_rotations),
                                        const_cast<float*>(d_shs), static_cast<cudaStream_t>(stream)), "assemble_backward");
    GSR_RANGE_POP();
    return rc;
}

int b200gsr_disparity_forward(int32_t B, int32_t N, const float* depth_alpha, const float* focal, float* out_disp,
                              void* stats, void* stream) {
    if (B < 0 || N < 0 || ((B > 0 && N > 0) && (!depth_alpha || !focal || !out_disp || !stats)))
        return fail(B200GSR_ERR_BAD_ARG, "bad disparity_forward arguments");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    return check_cuda(gsr_launch_disparity_fwd(B, N, depth_alpha, focal, out_disp, stats, ds->num_sms,
                                               static_cast<cudaStream_t>(stream)), "disparity_forward");
}

int b200gsr_disparity_backward(int32_t B, int32_t N, const float* depth_alpha, const float* focal, const float* g_disp,
                               const float* g_alpha, void* stats, float* d_depth_alpha, void* stream) {
    if (B < 0 || N < 0 || ((B > 0 && N > 0) && (!depth_alpha || !focal || !g_disp || !stats || !d_depth_alpha)))
        return fail(B200GSR_ERR_BAD_ARG, "bad disparity_backward arguments");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    return check_cuda(gsr_launch_disparity_bwd(B, N, depth_alpha, focal, g_disp, g_alpha, stats, d_depth_alpha,
                                               ds->num_sms, static_cast<cudaStream_t>(stream)), "disparity_backward");
}

#define GSR_ST(x) static_cast<cudaStream_t>(x)
int b200gsr_densify_stats(int32_t P, const float* viewspace_grad, const int32_t* radii, float* accum, float* denom,
                          float* max_radii2D, void* stream) {
    if (P < 0 || (P > 0 && (!viewspace_grad || !radii || !accum || !denom))) return fail(B200GSR_ERR_BAD_ARG, "bad densify_stats arguments");
    return check_cuda(gsr_densify_stats(P, viewspace_grad, radii, accum, denom, max_radii2D, GSR_ST(stream)), "densify_stats");
}
size_t b200gsr_densify_scratch_bytes(int32_t P) { return gsr_densify_scratch_bytes(P); }
int b200gsr_densify_plan(int32_t P, const float* accum, const float* denom, const float* scaling, const float* opacity,
                         float max_grad, float dense_extent, float min_opacity, float big_ws, float child_div,
                         void* scratch, uint32_t* totals5, void* stream) {
    if (P < 0 || !totals5 || (P > 0 && (!accum || !denom || !scaling || !opacity || !scratch)) || P > 0x0fffffff)
        return fail(B200GSR_ERR_BAD_ARG, "bad densify_plan arguments");
    return check_cuda(gsr_densify_plan(P, accum, denom, scaling, opacity, max_grad, dense_extent, min_opacity, big_ws,
                                       child_div, scratch, totals5, GSR_ST(stream)), "densify_plan");
}
int b200gsr_densify_map(int32_t P, int32_t N, const void* scratch, const uint32_t* totals5, int32_t* src_map,
                        int32_t* child_draw, void* stream) {
    if (P < 0 || N < 1 || (P > 0 && (!scratch || !totals5 || !src_map || !child_draw)))
        return fail(B200GSR_ERR_BAD_ARG, "bad densify_map arguments");
    return check_cuda(gsr_densify_map(P, N, scratch, totals5, src_map, child_draw, GSR_ST(stream)), "densify_map");
}
int b200gsr_compact_plan(int32_t P, const uint8_t* keep, void* scratch, int32_t* src_map, uint32_t* count, void* stream) {
    if (P < 0 || !count || (P > 0 && (!keep || !scratch || !src_map))) return fail(B200GSR_ERR_BAD_ARG, "bad compact_plan arguments");
    return check_cuda(gsr_compact_plan(P, keep, scratch, src_map, count, GSR_ST(stream)), "compact_plan");
}
int b200gsr_gather_rows(int32_t n_out, int32_t row_floats, const int32_t* src_map, const float* in, float* out,
                        int32_t zero_appended, void* stream) {
    if (n_out < 0 || row_floats < 0 || (n_out > 0 && row_floats > 0 && (!src_map || !in || !out)))
        return fail(B200GSR_ERR_BAD_ARG, "bad gather_rows arguments");
    return check_cuda(gsr_gather_rows(n_out, row_floats, src_map, in, out, zero_appended, GSR_ST(stream)), "gather_rows");
}
int b200gsr_split_children(int32_t n_out, int32_t first_child, float child_div, const int32_t* src_map,
                           const int32_t* child_draw, const float* xyz, const float* scaling, const float* rotation,
                           const float* z, float* xyz_out, float* scaling_out, void* stream) {
    if (n_out < 0 || first_child < 0 || (n_out > first_child && (!src_map || !child_draw || !xyz || !scaling || !rotation || !z || !xyz_out || !scaling_out)))
        return fail(B200GSR_ERR_BAD_ARG, "bad split_children arguments");
    return check_cuda(gsr_split_children(n_out, first_child, child_div, src_map, child_draw, xyz, scaling, rotation, z,
                                         xyz_out, scaling_out, GSR_ST(stream)), "split_children");
}
int b200gsr_kth_smallest(int32_t n, const float* v, uint32_t k, void* scratch, float* out, void* stream) {
    if (n < 0 || (n > 0 && (!v || !scratch || !out || k >= (uint32_t)n))) return fail(B200GSR_ERR_BAD_ARG, "bad kth_smallest arguments");
    DeviceState* ds = device_state();
    if (!ds) return fail(B200GSR_ERR_CUDA, "cannot query the current CUDA device");
    return check_cuda(gsr_kth_smallest(n, v, k, scratch, out, ds->num_sms, GSR_ST(stream)), "kth_smallest");
}

int b200gsr_debug_counters(unsigned long long* device_counters) {
    g_stats = device_counters;
    return B200GSR_OK;
}

size_t b200gsr_dist2_scratch_bytes(int32_t P) { return P < 0 ? 0 : gsr_knn_scratch_bytes(P, nullptr); }

int b200gsr_dist2_knn3(int32_t P, const float* points, float* out, void* scratch, size_t scratch_bytes,
                       void* stream) {
    if (P < 0 || (P > 0 && (!points || !out || !scratch)))
        return fail(B200GSR_ERR_BAD_ARG, "bad dist2_knn3 arguments");
    if (scratch_bytes < gsr_knn_scratch_bytes(P, nullptr))
        return fail(B200GSR_ERR_WORKSPACE, "dist2_knn3 scratch too small: %zu < %zu", scratch_bytes,
                    gsr_knn_scratch_bytes(P, nullptr));
    return check_cuda(gsr_launch_knn(P, points, out, static_cast<uint8_t*>(scratch), static_cast<cudaStream_t>(stream)),
                      "dist2_knn3");
}

int b200gsr_sh_grad_expand(int32_t P, int32_t M, int32_t sh_degree, int32_t num_views, const float* means3D,
                           const float* dcol, size_t view_stride, float* d_shs, void* stream) {
    if (P < 0 || M < 1 || num_views < 1 || num_views > 64 || sh_degree < 0 || sh_degree > 3 ||
        M < (sh_degree + 1) * (sh_degree + 1) || view_stride < 3 * (size_t)P + 3 || (P > 0 && (!means3D || !dcol || !d_shs)))
        return fail(B200GSR_ERR_BAD_ARG, "bad sh_grad_expand arguments");
    return check_cuda(gsr_launch_sh_grad_expand(P, M, sh_degree, num_views, means3D, dcol, view_stride, d_shs,
                                                static_cast<cudaStream_t>(stream)), "sh_grad_expand");
}

int b200gsr_mark_visible(int32_t P, const float* means3D, const float* viewmatrix,
                         const float* projmatrix, uint8_t* visible, void* stream) {
    if (P < 0 || (P > 0 && (!means3D || !viewmatrix || !visible)))
        return fail(B200GSR_ERR_BAD_ARG, "bad mark_visible arguments");
    return check_cuda(gsr_launch_mark_visible(P, means3D, viewmatrix, projmatrix, visible,
                                              static_cast<cudaStream_t>(stream)), "mark_visible");
}

}  // extern "C"
