// backward.cu -- gradients of a rendered whole frame with respect to the scene (lcgs_b200_render_backward).
// No reference counterpart: the reference renders only.  The derivatives themselves live in lcgs_grad.cuh.
//
//  * rebuild_records_kernel : the 48-byte blend records of the frame, rebuilt from the frame's own means_2d, conic
//    and colour and the scene's opacity (or alpha_consts) with the forward's write_record -- bit-identical to what
//    the forward's preprocess wrote, so the backward never depends on the context's workspace from the forward and
//    any number of frames may be rendered between a frame and its backward.
//  * blend_backward_kernel : one 128-thread CTA per tile in the forward's longest-first order, the forward's
//    geometry (four warps, 8x8 patch per warp, lane = pixels (x, y) and (x, y + 4)) and its round-based cp.async
//    staging with one barrier per round.  Each pixel replays the forward's front-to-back walk with the forward's
//    operations (blend_power, ex2-based alpha, T (1 - alpha) < 1e-4 stop), so it blends exactly the entries the
//    forward blended; the final colour C is read back from the image, and R_i . G = C . G - sum_{j<=i} w_j c_j . G
//    needs no reverse walk and no stored per-pixel state.  Per hit, each lane adds its two pixels' contributions to
//    the Gaussian's 9 values (mean x/y, conic, dL/dpower, colour), the warp reduces them with shuffles and three
//    lanes add the sums to the Gaussian's packed [12] float entry with one vector reduction each (RED.128): one
//    global atomic set per (patch, Gaussian) with a contribution.
//  * preprocess_backward_kernel : one thread per Gaussian; Gaussians with tiles_touched == 0 get zeros.  Recomputes
//    the forward's intermediates from the scene and chains the packed 2D gradient to pos / scale / rotq / sh /
//    opacity.
// Float atomics make the summation order, and so the last bits of the gradients, vary from run to run; the forward
// is untouched and stays bit-reproducible.
#include "common.cuh"
#include "lcgs_grad.cuh"

namespace lcgs_b200 {

namespace {

constexpr int kBwdThreads = 128;
constexpr int kBwdWarps   = kBwdThreads / 32;

__device__ __forceinline__ float4 bwd_lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

__device__ __forceinline__ float bwd_lds32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ void bwd_cp_async_16(uint32_t smem_addr, const void* gptr)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}

__device__ __forceinline__ void bwd_cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

// the forward's alpha: 2^(power * log2(e) + log2(opacity)) on MUFU.EX2 (blend.cu)
__device__ __forceinline__ float bwd_ex2_ftz(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

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

__global__ void __launch_bounds__(256)
    rebuild_records_kernel(int P, const float* __restrict__ means_2d, const float* __restrict__ conic,
                           const float* __restrict__ color, const float* __restrict__ opacity,
                           const float2* __restrict__ alpha_consts, const uint32_t* __restrict__ tiles_touched,
                           float4* __restrict__ records)
{
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P || __ldg(tiles_touched + i) == 0u) return;
    Splat2D s;
    s.px       = __ldg(means_2d + 2 * i);
    s.py       = __ldg(means_2d + 2 * i + 1);
    s.conic[0] = __ldg(conic + 3 * i);
    s.conic[1] = __ldg(conic + 3 * i + 1);
    s.conic[2] = __ldg(conic + 3 * i + 2);
    const float rgb[3] = { __ldg(color + 3 * i), __ldg(color + 3 * i + 1), __ldg(color + 3 * i + 2) };
    float       thr, l2op;
    if (alpha_consts) {
        const float2 k = __ldg(alpha_consts + i);
        thr = k.x; l2op = k.y;
    } else {
        const float op = __ldg(opacity + i);
        thr  = alpha_threshold(op);
        l2op = log2f(op);
    }
    write_record(records + (size_t)i * kRecordFloat4s, s, thr, l2op, rgb);
}

__global__ void __launch_bounds__(kBwdThreads)
    blend_backward_kernel(int W, int H, uint32_t gx, const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                          const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                          const float* __restrict__ img, const float* __restrict__ dl_dimg, float4* __restrict__ grad2d)
{
    __shared__ float4   s_rec[2][3][kBwdThreads];  // [buffer][plane][slot], planes as in the forward's blend
    __shared__ uint32_t s_id[2][kBwdThreads];     // [buffer][slot]: Gaussian index of the staged record
    __shared__ uint32_t s_cnt[2][kBwdWarps];

    const int      tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned FULL  = 0xFFFFFFFFu;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(&s_rec[0][0][0]);
    constexpr uint32_t kPlane = kBwdThreads * 16u, kBuf = 3u * kPlane;

    const uint32_t tile    = __ldg(order + blockIdx.x);
    const uint32_t tile_by = tile / gx, tile_bx = tile - tile_by * gx;
    const int tile_x0 = (int)tile_bx * 16, tile_y0 = (int)tile_by * 16;
    const int patch_x0 = tile_x0 + (warp & 1) * 8, patch_y0 = tile_y0 + (warp >> 1) * 8;
    const int px = patch_x0 + (lane & 7);
    const int pya = patch_y0 + (lane >> 3), pyb = pya + 4;
    const bool  in_a = px < W && pya < H, in_b = px < W && pyb < H;
    const float pxf = (float)px, pyaf = (float)pya, pybf = (float)pyb;  // no half-pixel offset (Q2)
    // the patch: culling is conservative, so any rectangle containing the pixels gives the forward's decisions
    const float wx0 = (float)patch_x0, wy0 = (float)patch_y0, wx1 = (float)(patch_x0 + 7), wy1 = (float)(patch_y0 + 7);

    const size_t plane = (size_t)W * (size_t)H;
    PixelGrad    pa, pb;
    {
        float C[3] = { 0.f, 0.f, 0.f }, G[3] = { 0.f, 0.f, 0.f };
        const size_t ia = (size_t)px + (size_t)W * (size_t)pya, ib = (size_t)px + (size_t)W * (size_t)pyb;
        if (in_a)
            for (int k = 0; k < 3; k++) { C[k] = __ldg(img + ia + k * plane); G[k] = __ldg(dl_dimg + ia + k * plane); }
        pa = pixel_grad_init(in_a, C, G);
        if (in_b)
            for (int k = 0; k < 3; k++) { C[k] = __ldg(img + ib + k * plane); G[k] = __ldg(dl_dimg + ib + k * plane); }
        else
            for (int k = 0; k < 3; k++) { C[k] = 0.f; G[k] = 0.f; }
        pb = pixel_grad_init(in_b, C, G);
    }

    const uint2    range   = __ldg(ranges + tile);
    const uint32_t len     = range.y > range.x ? range.y - range.x : 0u;
    const uint32_t nrounds = (len + kBwdThreads - 1) / kBwdThreads;

    // entry `lane` of the warp's 32 candidates goes to slot 31 - lane of the warp's segment (filled from the top, so
    // the walk from the highest hit bit meets the list in order), as in the forward
    auto stage = [&](uint32_t buf, bool valid, uint32_t id) {
        if (valid) {
            const uint32_t slot = (uint32_t)(warp * 32 + 31 - lane);
            const float4*  rec  = records + (size_t)id * kRecordFloat4s;
            const uint32_t addr = sbase + buf * kBuf + slot * 16u;
            bwd_cp_async_16(addr, rec);
            bwd_cp_async_16(addr + kPlane, rec + 1);
            bwd_cp_async_16(addr + 2u * kPlane, rec + 2);
            s_id[buf][slot] = id;
        }
        const unsigned v = __ballot_sync(FULL, valid);
        if (lane == 0) s_cnt[buf][warp] = __popc(v);
    };

    uint32_t next_id = 0;
    {
        const bool v0 = (uint32_t)tid < len;
        stage(0u, v0, v0 ? __ldg(point_list + range.x + tid) : 0u);
        if (kBwdThreads + (uint32_t)tid < len) next_id = __ldg(point_list + range.x + kBwdThreads + tid);
        bwd_cp_async_wait_all();
    }
    __syncthreads();

    for (uint32_t r = 0; r < nrounds; r++) {
        const uint32_t buf  = r & 1u;
        const uint32_t nidx = (r + 1u) * kBwdThreads + tid;
        if (r + 1u < nrounds) stage(buf ^ 1u, nidx < len, next_id);
        if (nidx + kBwdThreads < len) next_id = __ldg(point_list + range.x + nidx + kBwdThreads);

        if (!__all_sync(FULL, !(pa.T > 0.0f) && !(pb.T > 0.0f))) {
            const uint32_t abase = sbase + buf * kBuf;
#pragma unroll 1
            for (int seg = 0; seg < kBwdWarps; seg++) {
                const uint32_t cnt     = s_cnt[buf][seg];
                const uint32_t segbase = abase + seg * 512u;
                bool           hit     = false;
                if ((uint32_t)lane + cnt >= 32u) {
                    const float4 ga = bwd_lds128(segbase + lane * 16u);
                    const float4 gb = bwd_lds128(segbase + kPlane + lane * 16u);
                    const float  rx = bwd_lds32(segbase + 2u * kPlane + lane * 16u + 12u);
                    hit = !cull_rect_fast(ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.w, rx, wx0, wy0, wx1, wy1);
                }
                unsigned hits = __ballot_sync(FULL, hit);
                while (hits) {
                    const int      top  = 31 - __clz(hits);
                    const uint32_t addr = segbase + top * 16u;
                    hits ^= 1u << top;
                    const float4 ea = bwd_lds128(addr);
                    const float4 eb = bwd_lds128(addr + kPlane);
                    const float4 ec = bwd_lds128(addr + 2u * kPlane);
                    const float  rgb[3] = { ec.x, ec.y, ec.z };
                    float        g[kGrad2DValues];
#pragma unroll
                    for (int k = 0; k < kGrad2DValues; k++) g[k] = 0.0f;
                    // the forward's per-pixel operations (blend2_body's evaluate, scalar form)
                    const float dx  = ea.x - pxf;
                    const float dya = ea.y - pyaf, dyb = ea.y - pybf;
                    const float pwa = blend_power(ea.z, ea.w, eb.x, dx, dya);
                    const float pwb = blend_power(ea.z, ea.w, eb.x, dx, dyb);
                    const bool  oka = !(pwa > 0.0f) && !(pwa < eb.y);
                    const bool  okb = !(pwb > 0.0f) && !(pwb < eb.y);
                    const float ea_ = bwd_ex2_ftz(__fmaf_rn(pwa, 1.4426950408889634f, eb.z));
                    const float eb_ = bwd_ex2_ftz(__fmaf_rn(pwb, 1.4426950408889634f, eb.z));
                    bool contributed = blend_entry_grad(pa, oka, ea_, dx, dya, ea.z, ea.w, eb.x, rgb, g);
                    contributed |= blend_entry_grad(pb, okb, eb_, dx, dyb, ea.z, ea.w, eb.x, rgb, g);
                    if (__any_sync(FULL, contributed)) {
#pragma unroll
                        for (int k = 0; k < kGrad2DValues; k++)
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) g[k] += __shfl_xor_sync(FULL, g[k], o);
                        if (lane < 3) {
                            const uint32_t id = s_id[buf][seg * 32 + top];
                            const float4   v  = lane == 0 ? make_float4(g[0], g[1], g[2], g[3])
                                                : lane == 1 ? make_float4(g[4], g[5], g[6], g[7])
                                                            : make_float4(g[8], 0.0f, 0.0f, 0.0f);
                            atomicAdd(grad2d + (size_t)id * 3 + lane, v);  // RED.E.ADD.F32x4
                        }
                    }
                }
                if (__all_sync(FULL, !(pa.T > 0.0f) && !(pb.T > 0.0f))) break;
            }
        }
        bwd_cp_async_wait_all();
        if (__syncthreads_and(!(pa.T > 0.0f) && !(pb.T > 0.0f))) break;
    }
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
    float *         grad_means_2d, *grad_conic, *grad_color;
};

__global__ void __launch_bounds__(128) preprocess_backward_kernel(const __grid_constant__ PreprocessGradArgs a)
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

    rebuild_records_kernel<<<bwd_div_up(P, 256), 256, 0, s>>>(P, fr->means_2d, fr->conic, fr->color, sc->opacity,
                                                               reinterpret_cast<const float2*>(sc->alpha_consts),
                                                               fr->tiles_touched, records);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    // the tile schedule only: no count, so the context's device scalars (the last forward's) stay untouched
    if ((rc = launch_tile_order(ctx, fr->ranges, num_tiles, nullptr, 0, s))) return rc;
    blend_backward_kernel<<<(unsigned)num_tiles, kBwdThreads, 0, s>>>(W, H, gx, reinterpret_cast<const uint2*>(fr->ranges),
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
    preprocess_backward_kernel<<<bwd_div_up(P, 128), 128, 0, s>>>(a);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
