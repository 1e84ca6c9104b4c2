// project_sh (forward) and project_bwd (backward): the per-Gaussian streaming stages.
//
// Replaces upstream's preprocessCUDA / computeCov2DCUDA / preprocessCUDA-backward
// (comp-diff-gaussian-rasterization, un-vendored; functional spec: SURVEY.md App. A.1-A.5, A.7,
// restated in oracle/splat_ref.py::preprocess).  The SH basis follows
// /root/reference/utils/sh_utils.py:25-102, the covariance /root/reference/gs_renderer.py:124-157.
//
// Numerics contract: everything that decides an integer (depth bits, radius, tile rect) uses
// individually rounded fp32 ops (__fmul_rn/__fadd_rn/... are never FMA-contracted) in the order
// written in the oracle, so those integers are bit-exact against it.
#include "common.cuh"
#include <cuda_fp16.h>

#define MUL(a, b) __fmul_rn((a), (b))
#define ADD(a, b) __fadd_rn((a), (b))
#define SUB(a, b) __fsub_rn((a), (b))
#define DIV(a, b) __fdiv_rn((a), (b))
#define SQRT(a) __fsqrt_rn((a))

namespace {

#define SH_C0 0.28209479177387814f
#define SH_C1 0.4886025119029199f
#define SH_C2_0 1.0925484305920792f
#define SH_C2_1 -1.0925484305920792f
#define SH_C2_2 0.31539156525252005f
#define SH_C2_3 -1.0925484305920792f
#define SH_C2_4 0.5462742152960396f
#define SH_C3_0 -0.5900435899266435f
#define SH_C3_1 2.890611442640554f
#define SH_C3_2 -0.4570457994644658f
#define SH_C3_3 0.3731763325901154f
#define SH_C3_4 -0.4570457994644658f
#define SH_C3_5 1.445305721320277f
#define SH_C3_6 -0.5900435899266435f

struct Cam {
    float V[16];
    float F[16];
    float cam[3];
};

__device__ __forceinline__ void load_cam(const b200gsr_params& p, Cam& c) {
#pragma unroll
    for (int i = 0; i < 16; ++i) {
        c.V[i] = __ldg(p.viewmatrix + i);
        c.F[i] = __ldg(p.projmatrix + i);
    }
    c.cam[0] = __ldg(p.campos + 0);
    c.cam[1] = __ldg(p.campos + 1);
    c.cam[2] = __ldg(p.campos + 2);
}

// Geometry shared by forward and backward (bit-exact part).
struct Geo {
    float tx, ty, tz;        // view-space mean
    float hx, hy, hw, pw;    // clip-space, 1/(w+eps)
    float px, py;            // pixel mean
    float S[6];              // cov3D xx,xy,xz,yy,yz,zz
    float R[9], s[3];        // rotation, modified scales (only if !precomp)
    float cx, cy;            // clamped t.x, t.y
    bool in_x, in_y;
    float fx, fy;
    float J00, J02, J11, J12;
    float M0[3], M1[3], N0[3], N1[3];
    float a, b, c, det, det_inv;
};

__device__ __forceinline__ void geo_view(const Cam& C, float x, float y, float z, Geo& g) {
    g.tx = ADD(ADD(ADD(MUL(C.V[0], x), MUL(C.V[4], y)), MUL(C.V[8], z)), C.V[12]);
    g.ty = ADD(ADD(ADD(MUL(C.V[1], x), MUL(C.V[5], y)), MUL(C.V[9], z)), C.V[13]);
    g.tz = ADD(ADD(ADD(MUL(C.V[2], x), MUL(C.V[6], y)), MUL(C.V[10], z)), C.V[14]);
}

// raw per-Gaussian shape parameters, loadable ahead of the math (project_bwd issues these loads while
// its SH rows are still in flight)
struct RawShape {
    float s[3];
    float4 q;
    float cov[6];
};
__device__ __forceinline__ void load_shape(const float* __restrict__ scales, const float* __restrict__ rots,
                                           const float* __restrict__ cov3d, int i, RawShape& r) {
    if (cov3d != nullptr) {
#pragma unroll
        for (int k = 0; k < 6; ++k) r.cov[k] = __ldg(cov3d + 6 * (size_t)i + k);
    } else {
        r.s[0] = __ldg(scales + 3 * (size_t)i + 0);
        r.s[1] = __ldg(scales + 3 * (size_t)i + 1);
        r.s[2] = __ldg(scales + 3 * (size_t)i + 2);
        r.q = __ldg(reinterpret_cast<const float4*>(rots) + i);
    }
}

__device__ __forceinline__ void geo_rest(const Cam& C, const b200gsr_params& p, float x, float y,
                                         float z, bool has_cov, const RawShape& raw, Geo& g) {
    g.hx = ADD(ADD(ADD(MUL(C.F[0], x), MUL(C.F[4], y)), MUL(C.F[8], z)), C.F[12]);
    g.hy = ADD(ADD(ADD(MUL(C.F[1], x), MUL(C.F[5], y)), MUL(C.F[9], z)), C.F[13]);
    g.hw = ADD(ADD(ADD(MUL(C.F[3], x), MUL(C.F[7], y)), MUL(C.F[11], z)), C.F[15]);
    g.pw = DIV(1.0f, ADD(g.hw, 1e-7f));
    const float ndcx = MUL(g.hx, g.pw), ndcy = MUL(g.hy, g.pw);
    const float Wf = (float)p.image_width, Hf = (float)p.image_height;
    g.px = MUL(SUB(MUL(ADD(ndcx, 1.0f), Wf), 1.0f), 0.5f);
    g.py = MUL(SUB(MUL(ADD(ndcy, 1.0f), Hf), 1.0f), 0.5f);

    if (has_cov) {
#pragma unroll
        for (int k = 0; k < 6; ++k) g.S[k] = raw.cov[k];
    } else {
        const float mod = p.scale_modifier;
        g.s[0] = MUL(mod, raw.s[0]);
        g.s[1] = MUL(mod, raw.s[1]);
        g.s[2] = MUL(mod, raw.s[2]);
        const float4 q = raw.q;
        const float r = q.x, qx = q.y, qy = q.z, qz = q.w;
        g.R[0] = SUB(1.0f, MUL(2.0f, ADD(MUL(qy, qy), MUL(qz, qz))));
        g.R[1] = MUL(2.0f, SUB(MUL(qx, qy), MUL(r, qz)));
        g.R[2] = MUL(2.0f, ADD(MUL(qx, qz), MUL(r, qy)));
        g.R[3] = MUL(2.0f, ADD(MUL(qx, qy), MUL(r, qz)));
        g.R[4] = SUB(1.0f, MUL(2.0f, ADD(MUL(qx, qx), MUL(qz, qz))));
        g.R[5] = MUL(2.0f, SUB(MUL(qy, qz), MUL(r, qx)));
        g.R[6] = MUL(2.0f, SUB(MUL(qx, qz), MUL(r, qy)));
        g.R[7] = MUL(2.0f, ADD(MUL(qy, qz), MUL(r, qx)));
        g.R[8] = SUB(1.0f, MUL(2.0f, ADD(MUL(qx, qx), MUL(qy, qy))));
        float L[9];
#pragma unroll
        for (int r_ = 0; r_ < 3; ++r_)
#pragma unroll
            for (int c_ = 0; c_ < 3; ++c_) L[3 * r_ + c_] = MUL(g.R[3 * r_ + c_], g.s[c_]);
#define LDOT(i_, j_) ADD(ADD(MUL(L[3 * i_], L[3 * j_]), MUL(L[3 * i_ + 1], L[3 * j_ + 1])), \
                         MUL(L[3 * i_ + 2], L[3 * j_ + 2]))
        g.S[0] = LDOT(0, 0); g.S[1] = LDOT(0, 1); g.S[2] = LDOT(0, 2);
        g.S[3] = LDOT(1, 1); g.S[4] = LDOT(1, 2); g.S[5] = LDOT(2, 2);
#undef LDOT
    }

    const float limx = MUL(1.3f, p.tanfovx), limy = MUL(1.3f, p.tanfovy);
    g.fx = DIV(Wf, MUL(2.0f, p.tanfovx));
    g.fy = DIV(Hf, MUL(2.0f, p.tanfovy));
    const float txtz = DIV(g.tx, g.tz), tytz = DIV(g.ty, g.tz);
    g.in_x = (txtz >= -limx) && (txtz <= limx);
    g.in_y = (tytz >= -limy) && (tytz <= limy);
    g.cx = MUL(fminf(limx, fmaxf(-limx, txtz)), g.tz);
    g.cy = MUL(fminf(limy, fmaxf(-limy, tytz)), g.tz);
    const float tz2 = MUL(g.tz, g.tz);
    g.J00 = DIV(g.fx, g.tz);
    g.J02 = -DIV(MUL(g.fx, g.cx), tz2);
    g.J11 = DIV(g.fy, g.tz);
    g.J12 = -DIV(MUL(g.fy, g.cy), tz2);
    // Wr[i][k] = V[4k+i]
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        g.M0[k] = ADD(MUL(g.J00, C.V[4 * k + 0]), MUL(g.J02, C.V[4 * k + 2]));
        g.M1[k] = ADD(MUL(g.J11, C.V[4 * k + 1]), MUL(g.J12, C.V[4 * k + 2]));
    }
    const float Sg[9] = {g.S[0], g.S[1], g.S[2], g.S[1], g.S[3], g.S[4], g.S[2], g.S[4], g.S[5]};
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        g.N0[j] = ADD(ADD(MUL(g.M0[0], Sg[j]), MUL(g.M0[1], Sg[3 + j])), MUL(g.M0[2], Sg[6 + j]));
        g.N1[j] = ADD(ADD(MUL(g.M1[0], Sg[j]), MUL(g.M1[1], Sg[3 + j])), MUL(g.M1[2], Sg[6 + j]));
    }
    g.a = ADD(ADD(ADD(MUL(g.N0[0], g.M0[0]), MUL(g.N0[1], g.M0[1])), MUL(g.N0[2], g.M0[2])), 0.3f);
    g.b = ADD(ADD(MUL(g.N0[0], g.M1[0]), MUL(g.N0[1], g.M1[1])), MUL(g.N0[2], g.M1[2]));
    g.c = ADD(ADD(ADD(MUL(g.N1[0], g.M1[0]), MUL(g.N1[1], g.M1[1])), MUL(g.N1[2], g.M1[2])), 0.3f);
    g.det = SUB(MUL(g.a, g.c), MUL(g.b, g.b));
    g.det_inv = DIV(1.0f, g.det);
}

__device__ __forceinline__ int tile_coord(float v, int gmax) {
    float t = MUL(v, 0.0625f);
    if (isnan(t)) t = 0.0f;
    t = fminf(fmaxf(t, -1.0f), (float)gmax + 1.0f);
    int q = __float2int_rz(t);
    return min(gmax, max(0, q));
}

// ---- SH ----------------------------------------------------------------------------------
// SH coefficients are staged through shared memory with asynchronous copies (cp.async, no
// register round trip, all copies of a block in flight at once): a block of kBlock Gaussians owns
// kBlock rows of `stride` floats.  stride is a multiple of 4 with stride/4 odd, so rows are 16-B
// aligned and the per-thread LDS.128 row walks are bank-conflict free (8 lanes x 16 B hit 8
// distinct 4-bank groups).  Only rows of visible Gaussians are fetched.
constexpr int kBlock = 128;

__host__ __device__ __forceinline__ int sh_row_stride(int M) {
    int s4 = (3 * M + 3) / 4;
    if ((s4 & 1) == 0) ++s4;
    return 4 * s4;
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" :: "r"(smem_u32(smem_dst)), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// MT > 0: M known at compile time (16 = objects, 4 = scenes) -> the block's rows are one contiguous
// span of kBlock*3M floats that the threads copy as a flat sequence of 16-B units (perfectly
// coalesced, constant-divisor index math).  MT == 0: generic M (half a warp per row).
template <int MT, bool WAIT = true>
__device__ __forceinline__ void stage_sh_rows(const float* __restrict__ shs, int M, int nf, int g0, int P,
                                              const uint8_t* vis, float* buf, int stride) {
    const int nchunk = (nf + 3) >> 2;
    if (MT > 0 && ((3 * MT) & 3) == 0) {
        constexpr int q4 = (3 * (MT > 0 ? MT : 4)) / 4;   // 16-B units per row
        const float* base = shs + (size_t)g0 * 3 * MT;
#pragma unroll
        for (int it = 0; it < q4; ++it) {
            const int u = it * kBlock + threadIdx.x;
            const int row = u / q4, c4 = u - row * q4;
            if (c4 < nchunk && g0 + row < P && vis[row]) cp_async16(buf + row * stride + 4 * c4, base + 4 * u);
        }
    } else {
        const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
        const int hl = lane & 15, hsel = lane >> 4;
        const bool vec = ((3 * M) & 3) == 0;
        for (int it = 0; it < kBlock / 8; ++it) {
            const int row = it * 8 + w * 2 + hsel;          // 4 warps x 2 rows per iteration
            if (g0 + row < P && vis[row]) {
                const float* src = shs + (size_t)(g0 + row) * 3 * M;
                float* dst = buf + row * stride;
                if (vec) {
                    if (hl < nchunk) cp_async16(dst + 4 * hl, src + 4 * hl);
                } else {
                    for (int col = hl; col < nf; col += 16) cp_async4(dst + col, src + col);
                }
            }
        }
    }
    if (WAIT) cp_async_wait_all();
    else asm volatile("cp.async.commit_group;" ::: "memory");
}

// basis values for degree <= 3 at unit direction (x,y,z): utils/sh_utils.py:73-102
__device__ __forceinline__ void sh_basis(int deg, float x, float y, float z, float (&B)[16]) {
    B[0] = SH_C0;
#pragma unroll
    for (int k = 1; k < 16; ++k) B[k] = 0.0f;
    if (deg > 0) {
        B[1] = -SH_C1 * y; B[2] = SH_C1 * z; B[3] = -SH_C1 * x;
        if (deg > 1) {
            const float xx = x * x, yy = y * y, zz = z * z, xy = x * y, yz = y * z, xz = x * z;
            B[4] = SH_C2_0 * xy; B[5] = SH_C2_1 * yz; B[6] = SH_C2_2 * (2.0f * zz - xx - yy);
            B[7] = SH_C2_3 * xz; B[8] = SH_C2_4 * (xx - yy);
            if (deg > 2) {
                B[9] = SH_C3_0 * y * (3.0f * xx - yy);
                B[10] = SH_C3_1 * xy * z;
                B[11] = SH_C3_2 * y * (4.0f * zz - xx - yy);
                B[12] = SH_C3_3 * z * (2.0f * zz - 3.0f * xx - 3.0f * yy);
                B[13] = SH_C3_4 * x * (4.0f * zz - xx - yy);
                B[14] = SH_C3_5 * z * (xx - yy);
                B[15] = SH_C3_6 * x * (xx - 3.0f * yy);
            }
        }
    }
}

// colour = 0.5 + sum_k B[k]*sh[k][c]; the row is read as float4 chunks (f = 3k + c)
__device__ __forceinline__ void sh_color(const float (&B)[16], const float* row, int nf, float (&raw)[3]) {
    raw[0] = raw[1] = raw[2] = 0.5f;
    const float4* r4 = reinterpret_cast<const float4*>(row);
#pragma unroll
    for (int q = 0; q < 12; ++q) {
        if (4 * q < nf) {
            const float4 v = r4[q];
            const float vv[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int f = 4 * q + e;
                if (f < nf) raw[f % 3] = fmaf(B[f / 3], vv[e], raw[f % 3]);
            }
        }
    }
}

// =========================================================================================
// Forward: one Gaussian per thread, kBlock Gaussians per CTA.
// =========================================================================================
template <int MT>
__global__ void __launch_bounds__(kBlock)
project_sh_kernel(b200gsr_params p, const float* __restrict__ means3D,
                  const float* __restrict__ shs, const float* __restrict__ colors,
                  const float* __restrict__ opac, const float* __restrict__ scales,
                  const float* __restrict__ rots, const float* __restrict__ cov3d,
                  int32_t* __restrict__ radii, uint4* __restrict__ rectdepth,
                  GsrRec* __restrict__ geom, uint32_t* __restrict__ tile_count,
                  uint32_t* __restrict__ zero_words, int num_zero_words, float* __restrict__ dgeom,
                  int rec_base, int tile_row_off, int ntiles_total) {
    extern __shared__ __align__(16) float sh_buf[];
    __shared__ uint8_t vis_s[kBlock];
    const int g0 = blockIdx.x * kBlock;
    const int i = g0 + threadIdx.x;
    const bool active = i < p.P;
    // prologue (replaces a memset node): zero the work-queue + per-tile pair counters that the
    // count kernel launched right after this one accumulates into
    for (int zw = i; zw < num_zero_words; zw += gridDim.x * kBlock) zero_words[zw] = 0u;
    Cam C;
    load_cam(p, C);
    const GsrTileGrid grid = gsr_grid(p.image_height, p.image_width);

    Geo g;
    float x = 0.f, y = 0.f, z = 0.f;
    int radius = 0;
    int minx = 0, maxx = 0, miny = 0, maxy = 0;
    uint4 rd = make_uint4(0u, 0u, 0u, 0u);
    bool vis = false;
    if (active) {
        x = __ldg(means3D + 3 * (size_t)i); y = __ldg(means3D + 3 * (size_t)i + 1);
        z = __ldg(means3D + 3 * (size_t)i + 2);
        geo_view(C, x, y, z, g);
        rd.z = __float_as_uint(g.tz);
        if (g.tz > GSR_NEAR_Z) {
            // (hoisting these loads above the depth cull was measured: 0.0852 vs 0.0854 ms, no gain)
            RawShape raw;
            load_shape(scales, rots, cov3d, i, raw);
            geo_rest(C, p, x, y, z, cov3d != nullptr, raw, g);
            if (g.det != 0.0f) {
                const float mid = MUL(0.5f, ADD(g.a, g.c));
                const float sq = SQRT(fmaxf(SUB(MUL(mid, mid), g.det), 0.1f));
                const float lam = fmaxf(ADD(mid, sq), SUB(mid, sq));
                float rad_f = ceilf(MUL(3.0f, SQRT(lam)));
                if (isnan(rad_f)) rad_f = 0.0f;
                rad_f = fminf(fmaxf(rad_f, 0.0f), 1.0e9f);
                minx = tile_coord(SUB(g.px, rad_f), grid.gx);
                maxx = tile_coord(ADD(ADD(g.px, rad_f), 15.0f), grid.gx);
                miny = tile_coord(SUB(g.py, rad_f), grid.gy);
                maxy = tile_coord(ADD(ADD(g.py, rad_f), 15.0f), grid.gy);
                const int touched = (maxx - minx) * (maxy - miny);
                if (touched > 0) {
                    vis = true;
                    radius = (int)rad_f;
                    rd.x = (uint32_t)minx | ((uint32_t)miny << 16);
                    rd.y = (uint32_t)maxx | ((uint32_t)maxy << 16);
                    rd.w = (uint32_t)touched;
                }
            }
        }
        if (vis) {      // multi-view: this view's rows of the vertically stacked image
            rd.x += (uint32_t)tile_row_off << 16;
            rd.y += (uint32_t)tile_row_off << 16;
            miny += tile_row_off; maxy += tile_row_off;
        }
        radii[rec_base + i] = radius;
        rectdepth[rec_base + i] = rd;
    }
    const int stride = sh_row_stride(p.M);
    const int ncoef = (p.sh_degree + 1) * (p.sh_degree + 1);
    if (shs != nullptr) {
        vis_s[threadIdx.x] = vis;
        __syncthreads();
        stage_sh_rows<MT>(shs, p.M, 3 * ncoef, g0, p.P, vis_s, sh_buf, stride);
        __syncthreads();
    }
    if (!vis) return;

    // fallback binning only (tile grid too large for the smem multisplit): privatised global
    // tile counters; the RED atomics overlap the colour math below
    if (!gsr_use_multisplit(ntiles_total)) {
        uint32_t* cnt = tile_count + (size_t)(((rec_base + i) >> 5) & (GSR_COPIES - 1)) * ntiles_total;
        for (int ty = miny; ty < maxy; ++ty)
            for (int tx = minx; tx < maxx; ++tx) atomicAdd(cnt + ty * grid.gx + tx, 1u);
    }

    float rgb[3];
    if (shs != nullptr) {
        float dx = x - C.cam[0], dy = y - C.cam[1], dz = z - C.cam[2];
        float dn = sqrtf(dx * dx + dy * dy + dz * dz);
        if (dn == 0.0f) dn = 1.0f;
        dx /= dn; dy /= dn; dz /= dn;
        float B[16];
        sh_basis(p.sh_degree, dx, dy, dz, B);
        sh_color(B, sh_buf + threadIdx.x * stride, 3 * ncoef, rgb);
        rgb[0] = fmaxf(rgb[0], 0.0f); rgb[1] = fmaxf(rgb[1], 0.0f); rgb[2] = fmaxf(rgb[2], 0.0f);
    } else {
        rgb[0] = __ldg(colors + 3 * (size_t)i); rgb[1] = __ldg(colors + 3 * (size_t)i + 1);
        rgb[2] = __ldg(colors + 3 * (size_t)i + 2);
    }
    const float o = __ldg(opac + i);
    // conservative half extents of the region where alpha can reach 1/255
    float ex = -1.0f, ey = -1.0f;
    if (o * 255.0f > 1.0f) {
        const float tau2 = 2.0f * __logf(o * 255.0f) * 1.01f + 0.01f;
        ex = sqrtf(tau2 * g.a) * 1.003f + 0.05f;
        ey = sqrtf(tau2 * g.c) * 1.003f + 0.05f;
        if (!(ex == ex)) ex = 65504.0f * 2.0f;   // NaN -> never cull
        if (!(ey == ey)) ey = 65504.0f * 2.0f;
    }
    const __half2 eh = __floats2half2_rn(ex, ey);
    GsrRec rec;
    rec.px = g.px; rec.py = g.py;      // view-local pixel coordinates (the composite kernels evaluate view-locally too)
#ifdef GSR_EXACT_EXP
    rec.A = MUL(g.c, g.det_inv);                      // raw conic (x, y, z) as the oracle forms it
    rec.B = MUL(-g.b, g.det_inv);
    rec.C = MUL(g.a, g.det_inv);
#else
    rec.A = -0.5f * GSR_LOG2E * MUL(g.c, g.det_inv);
    rec.B = GSR_LOG2E * MUL(g.b, g.det_inv);          // -log2e * conic.y, conic.y = -b/det
    rec.C = -0.5f * GSR_LOG2E * MUL(g.a, g.det_inv);
#endif
    rec.opacity = o; rec.depth = g.tz; rec.idx = (uint32_t)(rec_base + i);
    rec.r = rgb[0]; rec.g = rgb[1]; rec.b = rgb[2];
    rec.ext = *reinterpret_cast<const uint32_t*>(&eh);
    float4* dst = reinterpret_cast<float4*>(geom + rec_base + i);
    const float4* src = reinterpret_cast<const float4*>(&rec);
    dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[2];
    if (dgeom != nullptr) {   // gradient accumulators of this (visible) Gaussian start at zero
        float4* dz = reinterpret_cast<float4*>(dgeom + 12 * (size_t)(rec_base + i));
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        dz[0] = z4; dz[1] = z4; dz[2] = z4;
    }
}

// =========================================================================================
// Backward: one Gaussian per thread.  dgeom[i] = 12 accumulated floats from composite_bwd:
//   0: sum g*(2A dx + B dy)   1: sum g*(2C dy + B dx)      (g = dL/dG * G, scaled conic)
//   2: sum g*dx*dx  3: sum g*dx*dy  4: sum g*dy*dy
//   5: sum G*dL/dalpha (dL/dopacity)   6..8: dL/drgb   9: dL/ddepth   10,11: unused
// =========================================================================================
// Register budget: since the parameter loads were hoisted above the SH wait (they overlap the cp.async
// staging), 8 CTAs/SM (64 registers) spills: measured 0.147 ms vs 0.120 ms at 6 CTAs/SM (80 registers)
// and 0.142 ms before the overlap.
template <int MT>
__global__ void __launch_bounds__(kBlock, 6)
project_bwd_kernel(b200gsr_params p, const float* __restrict__ means3D,
                   const float* __restrict__ shs, const float* __restrict__ colors,
                   const float* __restrict__ scales, const float* __restrict__ rots,
                   const float* __restrict__ cov3d, const int32_t* __restrict__ radii,
                   float* __restrict__ dgeom, uint32_t* __restrict__ bwd_queue,
                   int g_base, int g_end, int dsh_coefs, int rec_base, int accumulate,
                   float* __restrict__ d_means3D, float* __restrict__ d_means2D,
                   float* __restrict__ d_shs, float* __restrict__ d_colors,
                   float* __restrict__ d_opac, float* __restrict__ d_scales,
                   float* __restrict__ d_rots, float* __restrict__ d_cov3d) {
    extern __shared__ __align__(16) float sh_buf[];
    __shared__ uint8_t vis_s[kBlock];
    // this launch covers Gaussians [g_base, g_end); the launcher passes the whole view [0, P_view)
    const int g0 = g_base + blockIdx.x * kBlock;
    const int i = g0 + threadIdx.x;
    const bool active = i < g_end;
    const bool vis = active && (__ldg(radii + rec_base + i) > 0);
    const int nsh = 3 * dsh_coefs;          // floats per row of d_shs: 3*M (reference layout) or compact
    const int stride = sh_row_stride(p.M);
    const int deg = p.sh_degree;
    const int ncoef = (deg + 1) * (deg + 1);
    if (shs != nullptr) {
        vis_s[threadIdx.x] = vis;
        __syncthreads();
        stage_sh_rows<MT, false>(shs, p.M, 3 * ncoef, g0, g_end, vis_s, sh_buf, stride);   // issue only
    }
    // every other global load of this thread is issued while the SH rows are still in flight
    float x = 0.f, y = 0.f, z = 0.f;
    RawShape raw;
    float4 a0 = make_float4(0.f, 0.f, 0.f, 0.f), a1 = a0, a2 = a0;
    float4* dg = nullptr;
    if (vis) {
        x = __ldg(means3D + 3 * (size_t)i); y = __ldg(means3D + 3 * (size_t)i + 1); z = __ldg(means3D + 3 * (size_t)i + 2);
        load_shape(scales, rots, cov3d, i, raw);
        dg = reinterpret_cast<float4*>(dgeom + 12 * (size_t)(rec_base + i));
        a0 = dg[0]; a1 = dg[1]; a2 = dg[2];
    }
    if (shs != nullptr) {
        cp_async_wait_all();
        __syncthreads();
    }
    float dmean[3] = {0.f, 0.f, 0.f};
    float dm2[2] = {0.f, 0.f};
    float dop = 0.f;
    float dc3o[3] = {0.f, 0.f, 0.f};     // factored SH gradient (dsh_coefs < 0): dL/d(clamped colour), see below
    const bool factored = dsh_coefs < 0;
    float dsc[3] = {0.f, 0.f, 0.f};
    float drot[4] = {0.f, 0.f, 0.f, 0.f};
    float dcov[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
    float dcol[3] = {0.f, 0.f, 0.f};
    // composite_bwd (the previous kernel on the stream) has drained its work queue: reset it
    if (g_base == 0 && rec_base == 0 && blockIdx.x == 0 && threadIdx.x < GSR_NQUEUE) bwd_queue[threadIdx.x] = 0u;

    if (vis) {
        Cam C;
        load_cam(p, C);
        Geo g;
        geo_view(C, x, y, z, g);
        geo_rest(C, p, x, y, z, cov3d != nullptr, raw, g);
        // read-and-clear: the accumulators are zero again for the next backward over this `saved`
        const float4 z4 = make_float4(0.f, 0.f, 0.f, 0.f);
        dg[0] = z4; dg[1] = z4; dg[2] = z4;
        const float Wf = (float)p.image_width, Hf = (float)p.image_height;

        // ---- mean2D -------------------------------------------------------------------------
        const float dpx = GSR_PX_GRAD_SCALE * a0.x, dpy = GSR_PX_GRAD_SCALE * a0.y;   // dL/d(pixel mean)
        const float dndcx = dpx * 0.5f * Wf, dndcy = dpy * 0.5f * Hf;
        dm2[0] = dndcx; dm2[1] = dndcy;
        const float pw = g.pw, pw2 = pw * pw;
        const float mul1 = g.hx * pw2, mul2 = g.hy * pw2;
        dmean[0] = (C.F[0] * pw - C.F[3] * mul1) * dndcx + (C.F[1] * pw - C.F[3] * mul2) * dndcy;
        dmean[1] = (C.F[4] * pw - C.F[7] * mul1) * dndcx + (C.F[5] * pw - C.F[7] * mul2) * dndcy;
        dmean[2] = (C.F[8] * pw - C.F[11] * mul1) * dndcx + (C.F[9] * pw - C.F[11] * mul2) * dndcy;

        // ---- opacity, colour ----------------------------------------------------------------
        dop = a1.y;
        const float drgb[3] = {a1.z, a1.w, a2.x};
        const float ddepth = a2.y;

        // ---- conic -> cov2D -----------------------------------------------------------------
        const float ga = -0.5f * a0.z, gb = -a0.w, gc = -0.5f * a1.x;   // dL/d(conic a,b,c)
        const float ca = g.a, cb = g.b, cc = g.c;
        const float di2 = g.det_inv * g.det_inv;
        const float da = (-cc * cc * ga + cb * cc * gb - cb * cb * gc) * di2;
        const float db = (2.f * cb * cc * ga - (ca * cc + cb * cb) * gb + 2.f * ca * cb * gc) * di2;
        const float dc = (-cb * cb * ga + ca * cb * gb - ca * ca * gc) * di2;

        // ---- cov2D -> cov3D (full, unsymmetrised) and -> M ----------------------------------
        float Gs[9];
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 3; ++k)
                Gs[3 * j + k] = da * g.M0[j] * g.M0[k] + db * g.M0[j] * g.M1[k] + dc * g.M1[j] * g.M1[k];
        float dM0[3], dM1[3];
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            dM0[j] = 2.f * da * g.N0[j] + db * g.N1[j];
            dM1[j] = 2.f * dc * g.N1[j] + db * g.N0[j];
        }
        // M0k = J00*V[4k+0] + J02*V[4k+2] ; M1k = J11*V[4k+1] + J12*V[4k+2]
        float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            dJ00 += dM0[k] * C.V[4 * k + 0];
            dJ02 += dM0[k] * C.V[4 * k + 2];
            dJ11 += dM1[k] * C.V[4 * k + 1];
            dJ12 += dM1[k] * C.V[4 * k + 2];
        }
        const float tz = g.tz, itz = 1.0f / tz, itz2 = itz * itz, itz3 = itz2 * itz;
        const float dcx = -g.fx * itz2 * dJ02;
        const float dcy = -g.fy * itz2 * dJ12;
        float dtz = -g.fx * itz2 * dJ00 - g.fy * itz2 * dJ11 + 2.f * g.fx * g.cx * itz3 * dJ02 +
                    2.f * g.fy * g.cy * itz3 * dJ12;
        const float dtx = g.in_x ? dcx : 0.f;
        const float dty = g.in_y ? dcy : 0.f;
        dtz += ddepth;
        dmean[0] += C.V[0] * dtx + C.V[1] * dty + C.V[2] * dtz;
        dmean[1] += C.V[4] * dtx + C.V[5] * dty + C.V[6] * dtz;
        dmean[2] += C.V[8] * dtx + C.V[9] * dty + C.V[10] * dtz;

        if (cov3d != nullptr) {
            dcov[0] = Gs[0]; dcov[1] = Gs[1] + Gs[3]; dcov[2] = Gs[2] + Gs[6];
            dcov[3] = Gs[4]; dcov[4] = Gs[5] + Gs[7]; dcov[5] = Gs[8];
        } else {
            // Sigma = L L^T, L = R diag(s): dL = (Gs + Gs^T) L
            float L[9], dLm[9];
#pragma unroll
            for (int r_ = 0; r_ < 3; ++r_)
#pragma unroll
                for (int c_ = 0; c_ < 3; ++c_) L[3 * r_ + c_] = g.R[3 * r_ + c_] * g.s[c_];
#pragma unroll
            for (int r_ = 0; r_ < 3; ++r_)
#pragma unroll
                for (int c_ = 0; c_ < 3; ++c_) {
                    float acc = 0.f;
#pragma unroll
                    for (int k = 0; k < 3; ++k) acc += (Gs[3 * r_ + k] + Gs[3 * k + r_]) * L[3 * k + c_];
                    dLm[3 * r_ + c_] = acc;
                }
            float dR[9];
#pragma unroll
            for (int c_ = 0; c_ < 3; ++c_) {
                dsc[c_] = p.scale_modifier *
                          (dLm[c_] * g.R[c_] + dLm[3 + c_] * g.R[3 + c_] + dLm[6 + c_] * g.R[6 + c_]);
#pragma unroll
                for (int r_ = 0; r_ < 3; ++r_) dR[3 * r_ + c_] = dLm[3 * r_ + c_] * g.s[c_];
            }
            const float4 q = raw.q;
            const float r = q.x, qx = q.y, qy = q.z, qz = q.w;
            drot[0] = 2.f * (-qz * dR[1] + qy * dR[2] + qz * dR[3] - qx * dR[5] - qy * dR[6] + qx * dR[7]);
            drot[1] = 2.f * (qy * dR[1] + qz * dR[2] + qy * dR[3] - 2.f * qx * dR[4] - r * dR[5] +
                             qz * dR[6] + r * dR[7] - 2.f * qx * dR[8]);
            drot[2] = 2.f * (-2.f * qy * dR[0] + qx * dR[1] + r * dR[2] + qx * dR[3] + qz * dR[5] -
                             r * dR[6] + qz * dR[7] - 2.f * qy * dR[8]);
            drot[3] = 2.f * (-2.f * qz * dR[0] - r * dR[1] + qx * dR[2] + r * dR[3] - 2.f * qz * dR[4] +
                             qy * dR[5] + qx * dR[6] + qy * dR[7]);
        }

        // ---- colour -> SH (coefficients live in this thread's shared-memory row) -------------
        if (shs != nullptr) {
            float vx = x - C.cam[0], vy = y - C.cam[1], vz = z - C.cam[2];
            float dn = sqrtf(vx * vx + vy * vy + vz * vz);
            if (dn == 0.0f) dn = 1.0f;
            const float inv_n = 1.0f / dn;
            const float X = vx / dn, Y = vy / dn, Z = vz / dn;
            float* row = sh_buf + threadIdx.x * stride;
            const int nf = 3 * ncoef;
            float B[16], raw[3];
            sh_basis(deg, X, Y, Z, B);
            sh_color(B, row, nf, raw);
            float dc3[3];
#pragma unroll
            for (int c_ = 0; c_ < 3; ++c_) { dc3[c_] = (raw[c_] < 0.0f) ? 0.0f : drgb[c_]; dc3o[c_] = dc3[c_]; }
            // s_k = sum_c dL/drgb_c * sh[k][c]; then overwrite the row with dL/dsh (float4 chunks)
            float s[16];
#pragma unroll
            for (int k = 0; k < 16; ++k) s[k] = 0.f;
            float4* r4 = reinterpret_cast<float4*>(row);
#pragma unroll
            for (int q = 0; q < 12; ++q) {
                if (4 * q < nf) {
                    const float4 v = r4[q];
                    const float vv[4] = {v.x, v.y, v.z, v.w};
                    float o[4];
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int f = 4 * q + e;
                        o[e] = 0.f;
                        if (f < nf) {
                            s[f / 3] = fmaf(dc3[f % 3], vv[e], s[f / 3]);
                            o[e] = B[f / 3] * dc3[f % 3];
                        }
                    }
                    if (!factored) r4[q] = make_float4(o[0], o[1], o[2], o[3]);
                }
            }
            if (deg > 0) {
                float gx = -SH_C1 * s[3], gy = -SH_C1 * s[1], gz = SH_C1 * s[2];
                if (deg > 1) {
                    gx += SH_C2_0 * Y * s[4] + SH_C2_2 * (-2.f * X) * s[6] + SH_C2_3 * Z * s[7] + SH_C2_4 * 2.f * X * s[8];
                    gy += SH_C2_0 * X * s[4] + SH_C2_1 * Z * s[5] + SH_C2_2 * (-2.f * Y) * s[6] + SH_C2_4 * (-2.f * Y) * s[8];
                    gz += SH_C2_1 * Y * s[5] + SH_C2_2 * 4.f * Z * s[6] + SH_C2_3 * X * s[7];
                    if (deg > 2) {
                        const float xx = X * X, yy = Y * Y, zz = Z * Z;
                        gx += SH_C3_0 * 6.f * X * Y * s[9] + SH_C3_1 * Y * Z * s[10] + SH_C3_2 * (-2.f * X * Y) * s[11] +
                              SH_C3_3 * (-6.f * X * Z) * s[12] + SH_C3_4 * (4.f * zz - 3.f * xx - yy) * s[13] +
                              SH_C3_5 * 2.f * X * Z * s[14] + SH_C3_6 * (3.f * xx - 3.f * yy) * s[15];
                        gy += SH_C3_0 * (3.f * xx - 3.f * yy) * s[9] + SH_C3_1 * X * Z * s[10] +
                              SH_C3_2 * (4.f * zz - xx - 3.f * yy) * s[11] + SH_C3_3 * (-6.f * Y * Z) * s[12] +
                              SH_C3_4 * (-2.f * X * Y) * s[13] + SH_C3_5 * (-2.f * Y * Z) * s[14] +
                              SH_C3_6 * (-6.f * X * Y) * s[15];
                        gz += SH_C3_1 * X * Y * s[10] + SH_C3_2 * 8.f * Y * Z * s[11] +
                              SH_C3_3 * (6.f * zz - 3.f * xx - 3.f * yy) * s[12] + SH_C3_4 * 8.f * X * Z * s[13] +
                              SH_C3_5 * (xx - yy) * s[14];
                    }
                }
                // through d = v/|v|
                const float dotg = X * gx + Y * gy + Z * gz;
                dmean[0] += (gx - X * dotg) * inv_n;
                dmean[1] += (gy - Y * dotg) * inv_n;
                dmean[2] += (gz - Z * dotg) * inv_n;
            }
        } else {
            dcol[0] = drgb[0]; dcol[1] = drgb[1]; dcol[2] = drgb[2];
        }
    }

    // ---- dense writes (zeros for culled Gaussians).  `accumulate` (bit per output: 1 means3D, 2 opacity,
    // 4 sh/colour, 8 scales, 16 rotations, 32 cov3D) adds into the output instead: later views of a multi-view
    // backward that share the parameter with an earlier view.
#define GSR_OUT(ptr, val, bit) do { float* p_ = (ptr); *p_ = (accumulate & (bit)) ? *p_ + (val) : (val); } while (0)
    if (active) {
        GSR_OUT(d_means3D + 3 * (size_t)i, dmean[0], 1); GSR_OUT(d_means3D + 3 * (size_t)i + 1, dmean[1], 1);
        GSR_OUT(d_means3D + 3 * (size_t)i + 2, dmean[2], 1);
        d_means2D[3 * (size_t)i] = dm2[0]; d_means2D[3 * (size_t)i + 1] = dm2[1]; d_means2D[3 * (size_t)i + 2] = 0.f;
        GSR_OUT(d_opac + i, dop, 2);
        if (cov3d != nullptr) {
#pragma unroll
            for (int k = 0; k < 6; ++k) GSR_OUT(d_cov3d + 6 * (size_t)i + k, dcov[k], 32);
        } else {
            GSR_OUT(d_scales + 3 * (size_t)i, dsc[0], 8); GSR_OUT(d_scales + 3 * (size_t)i + 1, dsc[1], 8);
            GSR_OUT(d_scales + 3 * (size_t)i + 2, dsc[2], 8);
            float4* dr = reinterpret_cast<float4*>(d_rots) + i;
            float4 rv = make_float4(drot[0], drot[1], drot[2], drot[3]);
            if (accumulate & 16) { const float4 o = *dr; rv.x += o.x; rv.y += o.y; rv.z += o.z; rv.w += o.w; }
            *dr = rv;
        }
        if (shs == nullptr) {
            GSR_OUT(d_colors + 3 * (size_t)i, dcol[0], 4); GSR_OUT(d_colors + 3 * (size_t)i + 1, dcol[1], 4);
            GSR_OUT(d_colors + 3 * (size_t)i + 2, dcol[2], 4);
        }
    }
    if (shs != nullptr && factored) {
        // Factored SH gradient: dL/dsh[k][c] = basis_k(view direction) * dL/d(clamped colour)[c], so the three
        // colour gradients are all another rank needs to rebuild this view's [M, 3] rows (it knows the mean and
        // this view's camera centre): the multi-GPU payload drops from 3*M to 3 floats per Gaussian
        // (b200gsr_sh_grad_expand).  d_shs is a [P, 3] array here.
        if (active) {
            GSR_OUT(d_shs + 3 * (size_t)i, dc3o[0], 4); GSR_OUT(d_shs + 3 * (size_t)i + 1, dc3o[1], 4);
            GSR_OUT(d_shs + 3 * (size_t)i + 2, dc3o[2], 4);
        }
    } else if (shs != nullptr) {
        // drain the rows with coalesced stores (zeros for culled rows / inactive degrees)
        __syncthreads();
        const int nf = 3 * ncoef, nchunk = (nf + 3) >> 2;
        if (dsh_coefs != p.M) {
            // compact rows (only the active degree's coefficients, e.g. the NCCL payload at sh_degree 0):
            // the block's rows are one contiguous span of floats, written with coalesced 4-byte stores
            const int rows = min(kBlock, g_end - g0);
            float* base = d_shs + (size_t)g0 * nsh;
            for (int f = threadIdx.x; f < rows * nsh; f += kBlock) {
                const int row = f / nsh, col = f - row * nsh;
                const float val = (vis_s[row] && col < nf) ? sh_buf[row * stride + col] : 0.0f;
                base[f] = (accumulate & 4) ? base[f] + val : val;
            }
        } else if (MT > 0 && ((3 * MT) & 3) == 0) {
            constexpr int q4 = (3 * (MT > 0 ? MT : 4)) / 4;
            float* base = d_shs + (size_t)g0 * 3 * MT;
#pragma unroll
            for (int it = 0; it < q4; ++it) {
                const int u = it * kBlock + threadIdx.x;
                const int row = u / q4, c4 = u - row * q4;
                if (g0 + row < g_end) {
                    float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (c4 < nchunk && vis_s[row]) val = *reinterpret_cast<const float4*>(sh_buf + row * stride + 4 * c4);
                    if (accumulate & 4) {
                        const float4 o = ldg_f4(base + 4 * u);
                        val.x += o.x; val.y += o.y; val.z += o.z; val.w += o.w;
                    }
                    stg_na_f4(base + 4 * u, val);
                }
            }
        } else {
            const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
            const int hl = lane & 15, hsel = lane >> 4;
            const bool vec = (nsh & 3) == 0;
            for (int it = 0; it < kBlock / 8; ++it) {
                const int row = it * 8 + w * 2 + hsel;
                if (g0 + row >= g_end) continue;
                float* dst = d_shs + (size_t)(g0 + row) * nsh;
                const bool v = vis_s[row];
                if (vec) {
                    for (int q = hl; 4 * q < nsh; q += 16) {
                        float4 val = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (v && q < nchunk) val = *reinterpret_cast<const float4*>(sh_buf + row * stride + 4 * q);
                        if (accumulate & 4) {
                            const float4 o = ldg_f4(dst + 4 * q);
                            val.x += o.x; val.y += o.y; val.z += o.z; val.w += o.w;
                        }
                        stg_na_f4(dst + 4 * q, val);
                    }
                } else {
                    for (int col = hl; col < nsh; col += 16) {
                        const float val = (v && col < nf) ? sh_buf[row * stride + col] : 0.0f;
                        dst[col] = (accumulate & 4) ? dst[col] + val : val;
                    }
                }
            }
        }
    }
}

__global__ void mark_visible_kernel(int P, const float* __restrict__ means3D,
                                    const float* __restrict__ V, uint8_t* __restrict__ visible) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float x = means3D[3 * (size_t)i], y = means3D[3 * (size_t)i + 1], z = means3D[3 * (size_t)i + 2];
    const float tz = ADD(ADD(ADD(MUL(V[2], x), MUL(V[6], y)), MUL(V[10], z)), V[14]);
    visible[i] = tz > GSR_NEAR_Z;
}

}  // namespace

template <int MT>
static void launch_project_sh(const GsrFwdArgs& a, int P, size_t smem) {
    // multisplit path: counters + the single per-tile counter array are zeroed in the prologue
    // (api.cu issues a memset instead on the large-grid fallback, where this kernel counts itself)
    GsrTileGrid tg = gsr_grid(a.prm.image_height, a.prm.image_width);
    tg.gy = a.num_views * a.gy_view; tg.ntiles = tg.gx * tg.gy;      // the stacked image
    const int nzero = gsr_use_multisplit(tg.ntiles)
        ? (int)((a.sl.tile_count + (size_t)tg.ntiles * sizeof(uint32_t)) / sizeof(uint32_t)) : 0;
    project_sh_kernel<MT><<<(P + kBlock - 1) / kBlock, kBlock, smem, a.stream>>>(
        a.prm, a.means3D, a.shs, a.colors, a.opac, a.scales, a.rots, a.cov3d, a.radii,
        reinterpret_cast<uint4*>(a.scratch + a.sl.rectdepth),
        reinterpret_cast<GsrRec*>(a.saved + a.vl.geom),
        reinterpret_cast<uint32_t*>(a.scratch + a.sl.tile_count),
        reinterpret_cast<uint32_t*>(a.scratch), nzero,
        (a.flags & B200GSR_FWD_NO_BACKWARD) ? nullptr : reinterpret_cast<float*>(a.saved + a.vl.dgeom),
        a.view * a.P_view, a.view * a.gy_view, tg.ntiles);
}

cudaError_t gsr_launch_project(const GsrFwdArgs& a) {
    const int P = a.prm.P;
    if (P == 0) return cudaSuccess;
    const size_t smem = a.shs ? (size_t)kBlock * sh_row_stride(a.prm.M) * sizeof(float) : 0;
    if (a.shs && a.prm.M == 16) launch_project_sh<16>(a, P, smem);
    else if (a.shs && a.prm.M == 4) launch_project_sh<4>(a, P, smem);
    else launch_project_sh<0>(a, P, smem);
    return cudaGetLastError();
}

template <int MT>
static void launch_project_bwd(const GsrBwdArgs& a, size_t smem) {
    project_bwd_kernel<MT><<<(a.P_view + kBlock - 1) / kBlock, kBlock, smem, a.stream>>>(
        a.prm, a.means3D, a.shs, a.colors, a.scales, a.rots, a.cov3d, a.radii,
        reinterpret_cast<float*>(a.saved + a.vl.dgeom),
        reinterpret_cast<uint32_t*>(a.saved + a.vl.header) + GSR_H_BWD_QUEUE, 0, a.P_view,
        a.dsh_coefs > 0 ? a.dsh_coefs : (a.dsh_coefs < 0 ? -1 : a.prm.M), a.view * a.P_view, a.accumulate, a.d_means3D,
        a.d_means2D, a.d_shs,
        a.d_colors, a.d_opac, a.d_scales, a.d_rots, a.d_cov3d);
}

cudaError_t gsr_launch_project_bwd(const GsrBwdArgs& a) {
    if (a.P_view <= 0) return cudaSuccess;
    const size_t smem = a.shs ? (size_t)kBlock * sh_row_stride(a.prm.M) * sizeof(float) : 0;
    if (a.shs && a.prm.M == 16) launch_project_bwd<16>(a, smem);
    else if (a.shs && a.prm.M == 4) launch_project_bwd<4>(a, smem);
    else launch_project_bwd<0>(a, smem);
    return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------
// Rebuild the summed SH gradient of `nviews` views from their factored form (project_bwd with
// dsh_coefs < 0): d_shs[i][k][c] = sum_v basis_k(normalize(mean_i - cam_v)) * dcol_v[i][c].
// View v's record starts at dcol + v * stride floats: [P][3] colour gradients, then its camera centre (3 floats).
// The sum runs over v = 0 .. nviews-1 in order on every rank, so all ranks get bit-identical gradients.
// ---------------------------------------------------------------------------------------------
constexpr int kExpandViews = 64;
__global__ void __launch_bounds__(kBlock)
sh_grad_expand_kernel(int P, int M, int deg, int nviews, const float* __restrict__ means3D,
                      const float* __restrict__ dcol, size_t stride, float* __restrict__ d_shs) {
    extern __shared__ __align__(16) float ex_buf[];      // [kBlock][3*M] rows, drained with coalesced float4 stores
    __shared__ float cam_s[3 * kExpandViews];
    const int g0 = blockIdx.x * kBlock, i = g0 + threadIdx.x;
    const int ncoef = (deg + 1) * (deg + 1), nrow = 3 * M;
    for (int t = threadIdx.x; t < 3 * nviews; t += kBlock)
        cam_s[t] = __ldg(dcol + (size_t)(t / 3) * stride + 3 * (size_t)P + (t % 3));
    __syncthreads();
    float acc[16][3];
#pragma unroll
    for (int k = 0; k < 16; ++k) { acc[k][0] = 0.f; acc[k][1] = 0.f; acc[k][2] = 0.f; }
    if (i < P) {
        const float x = __ldg(means3D + 3 * (size_t)i), y = __ldg(means3D + 3 * (size_t)i + 1), z = __ldg(means3D + 3 * (size_t)i + 2);
        for (int v = 0; v < nviews; ++v) {
            const float* dc = dcol + (size_t)v * stride + 3 * (size_t)i;
            const float d0 = __ldg(dc), d1 = __ldg(dc + 1), d2 = __ldg(dc + 2);
            if (d0 == 0.f && d1 == 0.f && d2 == 0.f) continue;       // culled / clamped in this view
            const float vx = x - cam_s[3 * v], vy = y - cam_s[3 * v + 1], vz = z - cam_s[3 * v + 2];
            float dn = sqrtf(vx * vx + vy * vy + vz * vz);
            if (dn == 0.0f) dn = 1.0f;
            float B[16];
            sh_basis(deg, vx / dn, vy / dn, vz / dn, B);
#pragma unroll
            for (int k = 0; k < 16; ++k) {
                acc[k][0] = fmaf(B[k], d0, acc[k][0]); acc[k][1] = fmaf(B[k], d1, acc[k][1]); acc[k][2] = fmaf(B[k], d2, acc[k][2]);
            }
        }
    }
    float* row = ex_buf + (size_t)threadIdx.x * nrow;
#pragma unroll
    for (int k = 0; k < 16; ++k)
        if (k < M) { row[3 * k] = k < ncoef ? acc[k][0] : 0.f; row[3 * k + 1] = k < ncoef ? acc[k][1] : 0.f; row[3 * k + 2] = k < ncoef ? acc[k][2] : 0.f; }
    for (int k = 16; k < M; ++k) { row[3 * k] = 0.f; row[3 * k + 1] = 0.f; row[3 * k + 2] = 0.f; }
    __syncthreads();
    const int rows = min(kBlock, P - g0);
    const size_t nf = (size_t)rows * nrow;
    float* base = d_shs + (size_t)g0 * nrow;                 // 16-byte aligned when nrow*kBlock*4 % 16 == 0 (always: kBlock = 128)
    const size_t n4 = nf >> 2;
    for (size_t q = threadIdx.x; q < n4; q += kBlock)
        reinterpret_cast<float4*>(base)[q] = reinterpret_cast<const float4*>(ex_buf)[q];
    for (size_t f = (n4 << 2) + threadIdx.x; f < nf; f += kBlock) base[f] = ex_buf[f];
}

cudaError_t gsr_launch_sh_grad_expand(int P, int M, int deg, int nviews, const float* means3D, const float* dcol,
                                      size_t stride, float* d_shs, cudaStream_t s) {
    if (P == 0) return cudaSuccess;
    if (nviews < 1 || nviews > kExpandViews || deg < 0 || deg > 3 || M < (deg + 1) * (deg + 1)) return cudaErrorInvalidValue;
    const size_t smem = (size_t)kBlock * 3 * M * sizeof(float);
    if (smem > 48 * 1024) {
        cudaError_t e = cudaFuncSetAttribute(sh_grad_expand_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e != cudaSuccess) return e;
    }
    sh_grad_expand_kernel<<<(P + kBlock - 1) / kBlock, kBlock, smem, s>>>(P, M, deg, nviews, means3D, dcol, stride, d_shs);
    return cudaGetLastError();
}

cudaError_t gsr_launch_mark_visible(int P, const float* means3D, const float* view,
                                    const float* /*proj*/, uint8_t* visible, cudaStream_t s) {
    if (P == 0) return cudaSuccess;
    mark_visible_kernel<<<(P + 255) / 256, 256, 0, s>>>(P, means3D, view, visible);
    return cudaGetLastError();
}
