// backward.cu -- gradients of a rendered whole frame with respect to the scene (lcgs_b200_render_backward).
// No reference counterpart: the reference renders only.  The derivatives themselves live in lcgs_grad.cuh.
//
//  * the 48-byte blend records of the frame are rebuilt by the forward's build_records_kernel (preprocess.cu) from the
//    frame's own means_2d, conic and colour and the scene's opacity (or alpha_consts) -- bit-identical to what the
//    forward's preprocess wrote, so the backward never depends on the context's workspace from the forward and any
//    number of frames may be rendered between a frame and its backward.
//  * blend_backward_kernel : the forward's tile walk (walk_tile, blend_walk.cuh) in the forward's longest-first tile
//    order.  Each pixel replays the forward's front-to-back walk with the forward's operations (blend_power, ex2-based
//    alpha, T (1 - alpha) < 1e-4 stop), so it blends exactly the entries the forward blended; the final colour C is
//    read back from the image, and R_i . G = C . G - sum_{j<=i} w_j c_j . G needs no reverse walk and no stored
//    per-pixel state.  Per hit, each lane adds its two pixels' contributions to the Gaussian's 9 values (mean x/y,
//    conic, dL/dpower, colour), the warp reduces them with shuffles and three lanes add the sums to the Gaussian's
//    packed [12] float entry with one vector reduction each (RED.128): one global atomic set per (patch, Gaussian)
//    with a contribution.
//  * blend_backward_aux_kernel : the same walk (blend_backward_body<true>) when dL/d(alpha plane) or dL/d(depth plane)
//    is given: the planes are two more channels of the pixel's dot products, the candidate's view depth is staged with
//    its record by a fourth cp.async, and the warp reduces 10 values, the 10th (dL/dz) going to slot kG2Depth.
//  * preprocess_backward_kernel : one thread per Gaussian; Gaussians with tiles_touched == 0 get zeros.  Recomputes
//    the forward's intermediates from the scene and chains the packed 2D gradient to pos / scale / rotq / sh /
//    opacity (dL/dz through the view z).
// Float atomics make the summation order, and so the last bits of the gradients, vary from run to run; the forward
// is untouched and stays bit-reproducible.
#include "blend_walk.cuh"
#include "lcgs_grad.cuh"

namespace lcgs_b200 {

namespace {

struct GlobalShIn {
    const float* p;
    __device__ __forceinline__ float operator()(int k, int c) const { return __ldg(p + k * 3 + c); }
};

struct GlobalShOut {
    float* p;
    __device__ __forceinline__ void operator()(int k, int c, float v) const
    {
        if (p) p[k * 3 + c] = v;
    }
};

}  // namespace

// AUX (blend_backward_aux_kernel): the gradients of the frame's alpha and depth planes as well (lcgs_grad.cuh,
// PixelGradAux).  Each pixel also reads A, D and their gradients (a NULL gradient counts as 0); the candidate's view
// depth z = depth[id] is staged with its record by a fourth, 4-byte cp.async into s_z, as in blend2_aux_kernel
// (depth == NULL: no depth gradient, z = 0), and the warp reduces 10 values per hit, the 10th being dL/dz.
template <bool AUX>
__device__ __forceinline__ void blend_backward_body(const int tid, int W, int H, uint32_t gx, const uint2* __restrict__ ranges,
                                                    const uint32_t* __restrict__ order, const uint32_t* __restrict__ point_list,
                                                    const float4* __restrict__ records, const float* __restrict__ img,
                                                    const float* __restrict__ dl_dimg, const float* __restrict__ alpha,
                                                    const float* __restrict__ dplane, const float* __restrict__ dl_dalpha,
                                                    const float* __restrict__ dl_ddepth, const float* __restrict__ depth,
                                                    float4* __restrict__ grad2d)
{
    __shared__ float4   s_rec[2][3][kWalkThreads];  // [buffer][plane][slot], planes as in the record (common.cuh)
    __shared__ uint32_t s_cnt[2][kWalkWarps];
    __shared__ uint32_t s_id[2 * kWalkThreads];            // [buffer * 128 + slot]: Gaussian index of the staged record
    __shared__ float    s_z[AUX ? 2 * kWalkThreads : 1];  // [buffer * 128 + slot]: its view depth (AUX only)
    const uint32_t      zbase = AUX ? (uint32_t)__cvta_generic_to_shared(&s_z[0]) : 0u;
    constexpr int       NV    = AUX ? kGrad2DAuxValues : kGrad2DValues;

    const unsigned   FULL = 0xFFFFFFFFu;
    const TilePixels p    = tile_pixels(tid & 31, tid >> 5, order, gx, 0u);
    const bool       in_a = p.px < W && p.pya < H, in_b = p.px < W && p.pyb < H;
    const float      pxf = (float)p.px, pyaf = (float)p.pya, pybf = (float)p.pyb;  // no half-pixel offset (Q2)

    const size_t plane = (size_t)W * (size_t)H;
    PixelGradAux pa, pb;  // without AUX only .p is used
    {
        float C[3] = { 0.f, 0.f, 0.f }, G[3] = { 0.f, 0.f, 0.f };
        const size_t ia = (size_t)p.px + (size_t)W * (size_t)p.pya, ib = (size_t)p.px + (size_t)W * (size_t)p.pyb;
        // A, D, dL/dA, dL/dD of a pixel (AUX): a plane whose gradient is NULL does not enter
        auto planes = [&](bool in, size_t i, float* v) {
            v[0] = in && dl_dalpha ? __ldg(alpha + i) : 0.0f;
            v[1] = in && dl_ddepth ? __ldg(dplane + i) : 0.0f;
            v[2] = in && dl_dalpha ? __ldg(dl_dalpha + i) : 0.0f;
            v[3] = in && dl_ddepth ? __ldg(dl_ddepth + i) : 0.0f;
        };
        if (in_a)
            for (int k = 0; k < 3; k++) { C[k] = __ldg(img + ia + k * plane); G[k] = __ldg(dl_dimg + ia + k * plane); }
        if constexpr (AUX) {
            float v[4];
            planes(in_a, ia, v);
            pa = pixel_grad_aux_init(in_a, C, G, v[0], v[1], v[2], v[3]);
        } else {
            pa.p = pixel_grad_init(in_a, C, G);
        }
        if (in_b)
            for (int k = 0; k < 3; k++) { C[k] = __ldg(img + ib + k * plane); G[k] = __ldg(dl_dimg + ib + k * plane); }
        else
            for (int k = 0; k < 3; k++) { C[k] = 0.f; G[k] = 0.f; }
        if constexpr (AUX) {
            float v[4];
            planes(in_b, ib, v);
            pb = pixel_grad_aux_init(in_b, C, G, v[0], v[1], v[2], v[3]);
        } else {
            pb.p = pixel_grad_init(in_b, C, G);
        }
    }

    // The walk's cull box shrinks to the pixels still accumulating, as in the forward: the cull is conservative and a
    // finished pixel adds nothing in blend_entry_grad, so every pixel still meets the entries the forward blended.
    auto stage_id = [&](uint32_t entry, uint32_t id) {
        s_id[entry] = id;
        if constexpr (AUX)
            if (depth) cp_async_4(zbase + entry * 4u, depth + id);
    };
    auto no_consts = [] { return 0; };  // the scalar evaluation keeps no per-walk constants
    auto accumulate = [&](int, const float4& ea, const float4& eb, const float4& ec, uint32_t entry) {
        const float rgb[3] = { ec.x, ec.y, ec.z };
        float       g[NV];
#pragma unroll
        for (int k = 0; k < NV; k++) g[k] = 0.0f;
        // the forward's per-pixel operations (blend2_body's evaluate, scalar form)
        const float dx  = ea.x - pxf;
        const float dya = ea.y - pyaf, dyb = ea.y - pybf;
        const float pwa = blend_power(ea.z, ea.w, eb.x, dx, dya);
        const float pwb = blend_power(ea.z, ea.w, eb.x, dx, dyb);
        const bool  oka = !(pwa > 0.0f) && !(pwa < eb.y);
        const bool  okb = !(pwb > 0.0f) && !(pwb < eb.y);
        const float ea_ = ex2_ftz(__fmaf_rn(pwa, 1.4426950408889634f, eb.z));
        const float eb_ = ex2_ftz(__fmaf_rn(pwb, 1.4426950408889634f, eb.z));
        bool contributed;
        if constexpr (AUX) {
            const float z = depth ? lds32(zbase + entry * 4u) : 0.0f;
            contributed = blend_entry_grad_aux(pa, oka, ea_, dx, dya, ea.z, ea.w, eb.x, rgb, z, g);
            contributed |= blend_entry_grad_aux(pb, okb, eb_, dx, dyb, ea.z, ea.w, eb.x, rgb, z, g);
        } else {
            contributed = blend_entry_grad(pa.p, oka, ea_, dx, dya, ea.z, ea.w, eb.x, rgb, g);
            contributed |= blend_entry_grad(pb.p, okb, eb_, dx, dyb, ea.z, ea.w, eb.x, rgb, g);
        }
        if (__any_sync(FULL, contributed)) {
#pragma unroll
            for (int k = 0; k < NV; k++)
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) g[k] += __shfl_xor_sync(FULL, g[k], o);
            if (p.lane < 3) {
                const uint32_t id = s_id[entry];
                const float4   v  = p.lane == 0 ? make_float4(g[0], g[1], g[2], g[3])
                                    : p.lane == 1 ? make_float4(g[4], g[5], g[6], g[7])
                                                  : make_float4(g[8], AUX ? g[NV - 1] : 0.0f, 0.0f, 0.0f);
                atomicAdd(grad2d + (size_t)id * 3 + p.lane, v);  // RED.E.ADD.F32x4
            }
        }
    };
    walk_tile(tid, p, ranges, point_list, records, s_rec, s_cnt, pa.p.T, pb.p.T, stage_id, no_consts, accumulate);
}

__global__ void __launch_bounds__(kWalkThreads)
    blend_backward_kernel(int W, int H, uint32_t gx, const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                          const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                          const float* __restrict__ img, const float* __restrict__ dl_dimg, float4* __restrict__ grad2d)
{
    blend_backward_body<false>((int)threadIdx.x, W, H, gx, ranges, order, point_list, records, img, dl_dimg, nullptr,
                               nullptr, nullptr, nullptr, nullptr, grad2d);
}

// blend_backward_kernel plus the gradients of the alpha and depth planes (see blend_backward_body).  alpha / dplane:
// the frame's target_alpha / target_depth, read where dl_dalpha / dl_ddepth are non-NULL; depth: the frame's
// per-Gaussian view depth [P], non-NULL iff dl_ddepth is.
__global__ void __launch_bounds__(kWalkThreads)
    blend_backward_aux_kernel(int W, int H, uint32_t gx, const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                              const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                              const float* __restrict__ img, const float* __restrict__ dl_dimg,
                              const float* __restrict__ alpha, const float* __restrict__ dplane,
                              const float* __restrict__ dl_dalpha, const float* __restrict__ dl_ddepth,
                              const float* __restrict__ depth, float4* __restrict__ grad2d)
{
    blend_backward_body<true>((int)threadIdx.x, W, H, gx, ranges, order, point_list, records, img, dl_dimg, alpha, dplane,
                              dl_dalpha, dl_ddepth, depth, grad2d);
}

struct PreprocessGradArgs {
    int             P, sh_deg;
    const float*    pos;
    const float*    scale;
    const float*    rotq;
    const float*    sh;
    const float*    opacity;
    float           scale_modifier;
    ViewParams      vp;
    const uint32_t* tiles;
    const float4*   grad2d;
    float *         grad_pos, *grad_scale, *grad_rotq, *grad_sh, *grad_opacity;
    float *         grad_means_2d, *grad_conic, *grad_color, *grad_depth;
};

// 6 CTAs per SM: 80 registers, no spills.  Unbounded, the depth plane's dL/dz add in project_backward makes ptxas take
// 96 registers (5 CTAs per SM).
__global__ void __launch_bounds__(128, 6) preprocess_backward_kernel(const __grid_constant__ PreprocessGradArgs a)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.P) return;
    const int  feat = (a.sh_deg + 1) * (a.sh_deg + 1);
    float*     gsh  = a.grad_sh ? a.grad_sh + (size_t)i * feat * 3 : nullptr;
    if (__ldg(a.tiles + i) == 0u) {
        // discrete: a Gaussian no tile holds has no influence on the image
        for (int k = 0; k < 3; k++) {
            if (a.grad_pos) a.grad_pos[3 * i + k] = 0.0f;
            if (a.grad_scale) a.grad_scale[3 * i + k] = 0.0f;
            if (a.grad_conic) a.grad_conic[3 * i + k] = 0.0f;
            if (a.grad_color) a.grad_color[3 * i + k] = 0.0f;
        }
        if (a.grad_rotq)
            for (int k = 0; k < 4; k++) a.grad_rotq[4 * i + k] = 0.0f;
        if (a.grad_opacity) a.grad_opacity[i] = 0.0f;
        if (a.grad_means_2d) { a.grad_means_2d[2 * i] = 0.0f; a.grad_means_2d[2 * i + 1] = 0.0f; }
        if (a.grad_depth) a.grad_depth[i] = 0.0f;
        if (gsh)
            for (int k = 0; k < feat * 3; k++) gsh[k] = 0.0f;
        return;
    }
    float g2[kGrad2DFloats];
    {
        const float4 v0 = a.grad2d[3 * i], v1 = a.grad2d[3 * i + 1], v2 = a.grad2d[3 * i + 2];
        g2[0] = v0.x; g2[1] = v0.y; g2[2] = v0.z; g2[3] = v0.w;
        g2[4] = v1.x; g2[5] = v1.y; g2[6] = v1.z; g2[7] = v1.w;
        g2[8] = v2.x; g2[9] = v2.y; g2[10] = v2.z; g2[11] = v2.w;
    }
    if (a.grad_means_2d) { a.grad_means_2d[2 * i] = g2[kG2MeanX]; a.grad_means_2d[2 * i + 1] = g2[kG2MeanY]; }
    if (a.grad_depth) a.grad_depth[i] = g2[kG2Depth];
    for (int k = 0; k < 3; k++) {
        if (a.grad_conic) a.grad_conic[3 * i + k] = g2[kG2Conic0 + k];
        if (a.grad_color) a.grad_color[3 * i + k] = g2[kG2Red + k];
    }
    const float px = __ldg(a.pos + 3 * i), py = __ldg(a.pos + 3 * i + 1), pz = __ldg(a.pos + 3 * i + 2);
    float       dpos[3] = { 0.f, 0.f, 0.f }, dscale[3], drot[4];
    if (a.grad_pos || a.grad_scale || a.grad_rotq) {
        const float4 q = __ldg(reinterpret_cast<const float4*>(a.rotq) + i);
        project_backward(a.vp, a.scale_modifier, px, py, pz, __ldg(a.scale + 3 * i), __ldg(a.scale + 3 * i + 1),
                         __ldg(a.scale + 3 * i + 2), q.x, q.y, q.z, q.w, g2, dpos, dscale, drot);
    }
    if (a.grad_pos || gsh)
        sh_color_backward(a.sh_deg, a.vp.cam_pos, px, py, pz, GlobalShIn{ a.sh + (size_t)i * feat * 3 }, g2 + kG2Red,
                          GlobalShOut{ gsh }, dpos);
    if (a.grad_pos)
        for (int k = 0; k < 3; k++) a.grad_pos[3 * i + k] = dpos[k];
    if (a.grad_scale)
        for (int k = 0; k < 3; k++) a.grad_scale[3 * i + k] = dscale[k];
    if (a.grad_rotq)
        for (int k = 0; k < 4; k++) a.grad_rotq[4 * i + k] = drot[k];
    if (a.grad_opacity) {
        // dL/do = dL/dlog(o) / o (dalpha/do = alpha / o)
        const float op    = __ldg(a.opacity + i);
        a.grad_opacity[i] = op > 0.0f ? g2[kG2LogOp] / op : 0.0f;
    }
}

static inline uint32_t bwd_div_up(long a, long b) { return (uint32_t)((a + b - 1) / b); }

int launch_render_backward(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                           const lcgs_b200_frame* fr, const lcgs_b200_grad* gr, cudaStream_t s)
{
    const int P = sc->num_gaussians;
    if (P <= 0) return LCGS_B200_OK;
    const int      W = fr->width, H = fr->height;
    const uint32_t gx = (uint32_t)((W + 15) / 16), gy = (uint32_t)((H + 15) / 16);
    const int      num_tiles = (int)(gx * gy);  // whole frames only
    int            rc;
    if ((rc = ws_reserve(ctx, ctx->record_ws, (size_t)P * kRecordFloat4s * sizeof(float4)))) return rc;
    if ((rc = ws_reserve(ctx, ctx->grad_ws, (size_t)P * kGrad2DFloats * sizeof(float)))) return rc;
    float4* records = (float4*)ctx->record_ws.ptr;
    float4* grad2d  = (float4*)ctx->grad_ws.ptr;
    LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(grad2d, 0, (size_t)P * kGrad2DFloats * sizeof(float), s));

    if ((rc = launch_build_records(ctx, P, fr->means_2d, fr->conic, sc->opacity, sc->alpha_consts, fr->color,
                                   fr->tiles_touched, records, s)))
        return rc;
    // the tile schedule only: no count, so the context's device scalars (the last forward's) stay untouched
    if ((rc = launch_tile_order(ctx, fr->ranges, num_tiles, nullptr, 0, s))) return rc;
    if (gr->dl_dalpha || gr->dl_ddepth)
        blend_backward_aux_kernel<<<(unsigned)num_tiles, kWalkThreads, 0, s>>>(
            W, H, gx, reinterpret_cast<const uint2*>(fr->ranges), (const uint32_t*)ctx->tile_order_ws.ptr, fr->point_list,
            records, fr->target_img, gr->dl_dimg, fr->target_alpha, fr->target_depth, gr->dl_dalpha, gr->dl_ddepth,
            gr->dl_ddepth ? fr->depth : nullptr, grad2d);
    else
        blend_backward_kernel<<<(unsigned)num_tiles, kWalkThreads, 0, s>>>(W, H, gx, reinterpret_cast<const uint2*>(fr->ranges),
                                                                          (const uint32_t*)ctx->tile_order_ws.ptr, fr->point_list,
                                                                          records, fr->target_img, gr->dl_dimg, grad2d);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());

    PreprocessGradArgs a;
    a.P = P; a.sh_deg = sc->sh_deg;
    a.pos = sc->pos; a.scale = sc->scale; a.rotq = sc->rotq; a.sh = sc->sh; a.opacity = sc->opacity;
    a.scale_modifier = sc->scale_modifier;
    memcpy(&a.vp, vp, sizeof(ViewParams));
    a.tiles = fr->tiles_touched;
    a.grad2d = grad2d;
    a.grad_pos = gr->grad_pos; a.grad_scale = gr->grad_scale; a.grad_rotq = gr->grad_rotq; a.grad_sh = gr->grad_sh;
    a.grad_opacity = gr->grad_opacity;
    a.grad_means_2d = gr->grad_means_2d; a.grad_conic = gr->grad_conic; a.grad_color = gr->grad_color;
    a.grad_depth = gr->grad_depth;
    preprocess_backward_kernel<<<bwd_div_up(P, 128), 128, 0, s>>>(a);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
