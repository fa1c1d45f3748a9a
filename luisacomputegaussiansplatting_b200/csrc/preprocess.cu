// preprocess.cu -- stage 1: per-Gaussian work.
//
//  * preprocess_fused_kernel : SH colour (K1) + projection/EWA (K2) + conic/radius/tile rect (K3)
//    in one pass over the Gaussians, plus the packed 48-byte record the blend kernel gathers.
//    Replaces three DSL kernels with HBM round trips in between (sh_preprocessor.cpp:159-166,
//    gs_projector/shader.cpp:82-139, gs_tile_splatter/shader.cpp:102-163).
//  * sh_kernel / project_kernel / allocate_tiles_kernel / build_records_kernel : the same
//    arithmetic behind the reference's separate entry points.
//
// HBM-bound: algorithmic bytes per Gaussian = 40 (pos, scale, rotq) + 192 (SH, only when the
// Gaussian touches a tile) + outputs.  SH rows are fetched with block-cooperative, fully coalesced
// float4 loads predicated on "touches a tile", staged in padded shared memory (row stride 13
// float4 -> conflict-free LDS.128), so invisible/off-screen Gaussians never read their 192 bytes.
#include "common.cuh"

namespace lcgs_b200 {

struct PreprocessArgs {
    int          P, sh_deg;
    const float* pos;
    const float* scale;
    const float* rotq;
    const float* sh;
    const float* opacity;
    const float2* alpha_consts;  // optional per-scene (power threshold, log2 opacity), lcgs_b200_scene_prepare
    float        scale_modifier;
    ViewParams   vp;
    uint32_t     gx, gy, row0, row1;
    float*       means_2d;  // optional
    float*       depth;
    float*       conic;  // optional
    float*       color;  // optional
    int32_t*     radii;
    uint32_t*    tiles;
    float4*      records;
    uint2*       rects;  // packed tile rect of Gaussians that touch a tile: (x0 | y0<<16, w | h<<16)
};

constexpr int kPreThreads = 128;
constexpr int kShRowF4    = 12;  // 16 coefficients x RGB = 48 floats = 12 float4
constexpr int kShRowPad   = 13;  // padded row stride in float4

struct RegSh {
    const float* r;
    __device__ __forceinline__ float operator()(int k, int c) const { return r[k * 3 + c]; }
};

struct GlobalSh {
    const float* p;
    __device__ __forceinline__ float operator()(int k, int c) const { return __ldg(p + k * 3 + c); }
};

// The alpha-test constants depend on the opacity alone.  Computing the threshold is a binary64 search
// (alpha_threshold(), ~25 % of the fused kernel's issue slots), so a caller that renders many frames of one
// scene computes them once (lcgs_b200_scene_prepare) and passes them in lcgs_b200_scene::alpha_consts.
__global__ void __launch_bounds__(256) scene_prepare_kernel(int P, const float* __restrict__ opacity, float2* __restrict__ consts)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float op = __ldg(opacity + i);
    consts[i]      = make_float2(alpha_threshold(op), log2f(op));
}

// HAS_CONSTS: read (threshold, log2 opacity) from the per-scene array instead of deriving them from the opacity
template <bool HAS_CONSTS>
__global__ void __launch_bounds__(kPreThreads) preprocess_fused_kernel(const __grid_constant__ PreprocessArgs a)
{
    // Every warp works on its own 32 Gaussians and its own slice of shared memory: no block-wide
    // barrier, so a warp waiting for its SH rows never holds up the others.
    __shared__ float4 s_sh[kPreThreads * kShRowPad];

    const int      t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned FULL = 0xFFFFFFFFu;
    const long     w0   = (long)blockIdx.x * kPreThreads + warp * 32;  // first Gaussian of this warp
    const long     i    = w0 + lane;
    float4* const  w_sh = s_sh + warp * 32 * kShRowPad;

    // ---- phase 1: geometry ----------------------------------------------------------------
    float   px = 0.f, py = 0.f, pz = 0.f, thr = 0.f, l2op = 0.f;
    Splat2D s;
    s.tiles   = 0;
    bool need = false;
    if (i < a.P) {
        // opacity is only needed by Gaussians that touch a tile, but a predicated 4-byte load costs a
        // whole 32-byte sector per Gaussian; unconditionally the warp reads 128 contiguous bytes
        if (HAS_CONSTS) {
            const float2 k = __ldg(a.alpha_consts + i);
            thr = k.x; l2op = k.y;
        } else {
            l2op = __ldg(a.opacity + i);  // the opacity itself until phase 3
        }
        px = __ldg(a.pos + 3 * i);
        py = __ldg(a.pos + 3 * i + 1);
        pz = __ldg(a.pos + 3 * i + 2);
        const ViewPoint pv = view_transform(a.vp, px, py, pz);
        if (pv.visible) {
            const float  s0 = __ldg(a.scale + 3 * i), s1 = __ldg(a.scale + 3 * i + 1), s2 = __ldg(a.scale + 3 * i + 2);
            const float4 q  = __ldg(reinterpret_cast<const float4*>(a.rotq) + i);
            float        cov[3];
            ewa_cov2d(a.vp, pv, a.scale_modifier, s0, s1, s2, q.x, q.y, q.z, q.w, cov);
            s = splat_from_cov(pv.ndc_x, pv.ndc_y, cov, a.vp.width, a.vp.height, a.gx, a.gy, a.row0, a.row1);
            // depth, tile counts and rects are read again within microseconds (scan, emission): normal stores.  radii,
            // means_2d, conic and colour are outputs nothing in the frame reads back (the blend gathers the packed
            // records): streaming stores keep them from evicting the former from L2.
            a.depth[i] = pv.z;
            __stcs(a.radii + i, s.radius);
            a.tiles[i] = s.tiles;
            if (a.means_2d) __stcs(reinterpret_cast<float2*>(a.means_2d) + i, make_float2(s.px, s.py));
            if (a.conic) {
                __stcs(a.conic + 3 * i, s.conic[0]);
                __stcs(a.conic + 3 * i + 1, s.conic[1]);
                __stcs(a.conic + 3 * i + 2, s.conic[2]);
            }
            need = s.tiles > 0u;
            if (need && a.rects)
                a.rects[i] = make_uint2(s.rect.x0 | (s.rect.y0 << 16), (s.rect.x1 - s.rect.x0) | ((s.rect.y1 - s.rect.y0) << 16));
        } else {
            // defined behaviour for near-culled Gaussians (the reference leaves stale data, Q6)
            a.depth[i] = 0.0f;
            __stcs(a.radii + i, 0);
            a.tiles[i] = 0u;
            if (a.means_2d) __stcs(reinterpret_cast<float2*>(a.means_2d) + i, make_float2(0.f, 0.f));
            if (a.conic) {
                __stcs(a.conic + 3 * i, 0.f);
                __stcs(a.conic + 3 * i + 1, 0.f);
                __stcs(a.conic + 3 * i + 2, 0.f);
            }
        }
    }
    const unsigned need_mask = __ballot_sync(FULL, need);
    if (need_mask == 0u) return;

    // ---- phase 2: coalesced, predicated SH fetch into padded shared memory -------------------
    // The warp's 32 rows are one contiguous 6 KB run; lane l copies 16-byte pieces l, l+32, ... of it
    // with cp.async (LDGSTS: no register staging, all 12 requests of a lane in flight at once), but
    // only the pieces of rows whose Gaussian touches a tile.
    if (a.sh_deg == 3) {
        const float4*  src   = reinterpret_cast<const float4*>(a.sh) + w0 * kShRowF4;
        const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(w_sh);
#pragma unroll
        for (int j = 0; j < kShRowF4; j++) {
            const int idx = j * 32 + lane;
            const int g   = idx / kShRowF4;
            const int c   = idx - g * kShRowF4;
            if ((need_mask >> g) & 1u)  // implies w0 + g < P
                asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sbase + (uint32_t)(g * kShRowPad + c) * 16u),
                             "l"(src + idx)
                             : "memory");
        }
        asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
        __syncwarp();
    }

    // ---- phase 3: colour + blend record ------------------------------------------------------
    if (need) {
        float rgb[3];
        if (a.sh_deg == 3) {
            float r[48];
#pragma unroll
            for (int k = 0; k < kShRowF4; k++) {
                const float4 q = w_sh[lane * kShRowPad + k];
                r[4 * k] = q.x; r[4 * k + 1] = q.y; r[4 * k + 2] = q.z; r[4 * k + 3] = q.w;
            }
            sh_color(3, a.vp.cam_pos, px, py, pz, RegSh{ r }, rgb);
        } else {
            const int feat = (a.sh_deg + 1) * (a.sh_deg + 1);
            sh_color(a.sh_deg, a.vp.cam_pos, px, py, pz, GlobalSh{ a.sh + (size_t)i * feat * 3 }, rgb);
        }
        if (a.color) {
            __stcs(a.color + 3 * i, rgb[0]);
            __stcs(a.color + 3 * i + 1, rgb[1]);
            __stcs(a.color + 3 * i + 2, rgb[2]);
        }
        if (!HAS_CONSTS) {
            thr  = alpha_threshold(l2op);
            l2op = log2f(l2op);
        }
        write_record(a.records + (size_t)i * kRecordFloat4s, s, thr, l2op, rgb);
    }
}

// ---- the reference's separate passes -----------------------------------------------------------

__global__ void __launch_bounds__(256) sh_kernel(int P, int deg, float cx, float cy, float cz, const float* __restrict__ pos,
                                                 const float* __restrict__ sh, float* __restrict__ color)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const float cam[3] = { cx, cy, cz };
    const int   feat   = (deg + 1) * (deg + 1);
    float       rgb[3];
    sh_color(deg, cam, __ldg(pos + 3 * i), __ldg(pos + 3 * i + 1), __ldg(pos + 3 * i + 2),
             GlobalSh{ sh + (size_t)i * feat * 3 }, rgb);
    color[3 * i]     = rgb[0];
    color[3 * i + 1] = rgb[1];
    color[3 * i + 2] = rgb[2];
}

__global__ void __launch_bounds__(256)
    project_kernel(int P, const float* __restrict__ pos, const float* __restrict__ scale, const float* __restrict__ rotq,
                   float scale_modifier, const __grid_constant__ ViewParams vp, float* __restrict__ means_2d,
                   float* __restrict__ depth, float* __restrict__ covs_2d)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const ViewPoint pv = view_transform(vp, __ldg(pos + 3 * i), __ldg(pos + 3 * i + 1), __ldg(pos + 3 * i + 2));
    float           cov[3] = { 0.f, 0.f, 0.f };
    float           d = 0.f, nx = 0.f, ny = 0.f;
    if (pv.visible) {
        ewa_cov2d(vp, pv, scale_modifier, __ldg(scale + 3 * i), __ldg(scale + 3 * i + 1), __ldg(scale + 3 * i + 2),
                  __ldg(rotq + 4 * i), __ldg(rotq + 4 * i + 1), __ldg(rotq + 4 * i + 2), __ldg(rotq + 4 * i + 3), cov);
        d  = pv.z;
        nx = pv.ndc_x;
        ny = pv.ndc_y;
    }
    depth[i]            = d;
    means_2d[2 * i]     = nx;
    means_2d[2 * i + 1] = ny;
    covs_2d[3 * i]      = cov[0];
    covs_2d[3 * i + 1]  = cov[1];
    covs_2d[3 * i + 2]  = cov[2];
}

__global__ void __launch_bounds__(256)
    allocate_tiles_kernel(int P, int W, int H, uint32_t gx, uint32_t gy, uint32_t row0, uint32_t row1,
                          const float* __restrict__ depth, float* __restrict__ means_2d, float* __restrict__ covs_2d,
                          uint32_t* __restrict__ tiles_touched, int32_t* __restrict__ radii)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    int32_t  radius = 0;
    uint32_t tiles  = 0;
    if (!(depth[i] < 0.2f)) {
        const float   cov[3] = { covs_2d[3 * i], covs_2d[3 * i + 1], covs_2d[3 * i + 2] };
        const Splat2D s      = splat_from_cov(means_2d[2 * i], means_2d[2 * i + 1], cov, W, H, gx, gy, row0, row1);
        radius               = s.radius;
        tiles                = s.tiles;
        covs_2d[3 * i]       = s.conic[0];
        covs_2d[3 * i + 1]   = s.conic[1];
        covs_2d[3 * i + 2]   = s.conic[2];
        means_2d[2 * i]      = s.px;
        means_2d[2 * i + 1]  = s.py;
    }
    radii[i]         = radius;
    tiles_touched[i] = tiles;
}

// Packs the reference-layout buffers (after allocate_tiles) into blend records.
__global__ void __launch_bounds__(256)
    build_records_kernel(int P, const float* __restrict__ means_2d, const float* __restrict__ conic,
                         const float* __restrict__ opacity, const float* __restrict__ color,
                         const uint32_t* __restrict__ tiles_touched, float4* __restrict__ records)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    if (tiles_touched && tiles_touched[i] == 0u) return;
    Splat2D s;
    s.px       = means_2d[2 * i];
    s.py       = means_2d[2 * i + 1];
    s.conic[0] = conic[3 * i];
    s.conic[1] = conic[3 * i + 1];
    s.conic[2] = conic[3 * i + 2];
    const float rgb[3] = { color[3 * i], color[3 * i + 1], color[3 * i + 2] };
    const float op = opacity[i];
    write_record(records + (size_t)i * kRecordFloat4s, s, alpha_threshold(op), log2f(op), rgb);
}

// ---- launchers -------------------------------------------------------------------------------

static inline uint32_t div_up(long a, long b) { return (uint32_t)((a + b - 1) / b); }

int launch_preprocess_fused(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                            const lcgs_b200_frame* fr, float4* records, uint2* rects, cudaStream_t s)
{
    const int P = sc->num_gaussians;
    if (P <= 0) return LCGS_B200_OK;
    PreprocessArgs a;
    a.P = P; a.sh_deg = sc->sh_deg;
    a.pos = sc->pos; a.scale = sc->scale; a.rotq = sc->rotq; a.sh = sc->sh; a.opacity = sc->opacity;
    a.alpha_consts = reinterpret_cast<const float2*>(sc->alpha_consts);
    a.scale_modifier = sc->scale_modifier;
    static_assert(sizeof(ViewParams) == sizeof(lcgs_b200_view_params), "view params layout");
    memcpy(&a.vp, vp, sizeof(ViewParams));
    a.gx   = (uint32_t)((fr->width + 15) / 16);
    a.gy   = (uint32_t)((fr->height + 15) / 16);
    a.row0 = (uint32_t)fr->tile_row_begin;
    a.row1 = fr->tile_row_end < 0 ? a.gy : (uint32_t)fr->tile_row_end;
    a.means_2d = fr->means_2d; a.depth = fr->depth; a.conic = fr->conic; a.color = fr->color;
    a.radii = fr->radii; a.tiles = fr->tiles_touched; a.records = records; a.rects = rects;
    if (a.alpha_consts) preprocess_fused_kernel<true><<<div_up(P, kPreThreads), kPreThreads, 0, s>>>(a);
    else preprocess_fused_kernel<false><<<div_up(P, kPreThreads), kPreThreads, 0, s>>>(a);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_scene_prepare(lcgs_b200_ctx* ctx, int P, const float* opacity, float* consts, cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    scene_prepare_kernel<<<div_up(P, 256), 256, 0, s>>>(P, opacity, reinterpret_cast<float2*>(consts));
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_sh(lcgs_b200_ctx* ctx, int P, int deg, const float* cam_pos, const float* pos, const float* sh, float* color,
              cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    sh_kernel<<<div_up(P, 256), 256, 0, s>>>(P, deg, cam_pos[0], cam_pos[1], cam_pos[2], pos, sh, color);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_project(lcgs_b200_ctx* ctx, int P, const float* pos, const float* scale, const float* rotq,
                   float scale_modifier, const ViewParams& vp, float* means_2d, float* depth, float* covs_2d,
                   cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    project_kernel<<<div_up(P, 256), 256, 0, s>>>(P, pos, scale, rotq, scale_modifier, vp, means_2d, depth, covs_2d);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_allocate_tiles(lcgs_b200_ctx* ctx, int P, int W, int H, const float* depth, float* means_2d, float* covs_2d,
                          uint32_t* tiles_touched, int32_t* radii, int row0, int row1, cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    const uint32_t gx = (uint32_t)((W + 15) / 16), gy = (uint32_t)((H + 15) / 16);
    allocate_tiles_kernel<<<div_up(P, 256), 256, 0, s>>>(P, W, H, gx, gy, (uint32_t)row0,
                                                         row1 < 0 ? gy : (uint32_t)row1, depth, means_2d, covs_2d,
                                                         tiles_touched, radii);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_build_records(lcgs_b200_ctx* ctx, int P, const float* means_2d, const float* conic, const float* opacity,
                         const float* color, const uint32_t* tiles_touched, float4* records, cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    build_records_kernel<<<div_up(P, 256), 256, 0, s>>>(P, means_2d, conic, opacity, color, tiles_touched, records);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
