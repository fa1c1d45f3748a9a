// blend.cu -- stage 5b: per-tile front-to-back alpha blending.
// Replaces m_forward_render_shader (lcgs/src/gs_tile_splatter/shader.cpp:171-288).
//
// The tile walk -- one 128-thread CTA per 16x16 tile, an 8x8 patch per warp, two pixels per lane, rounds of 128 records
// staged with cp.async, each segment culled against the warp's unfinished pixels -- is walk_tile() (blend_walk.cuh),
// shared with the blend backward; this file adds the per-hit evaluation and the epilogue.  The cull is conservative
// with respect to the per-pixel evaluation: on the C3 scene 42 % of the (Gaussian, tile) instances binned by the
// reference's loose rect never touch their tile, and the reference evaluates all of them for 256 pixels.
// A Gaussian that hits a patch is fetched once for its 64 pixels with broadcast LDS.128, and the arithmetic of a lane's
// pixel pair runs on Blackwell's packed FP32 instructions (FADD2 / FMUL2 / FFMA2: two IEEE binary32 operations per lane
// and issue slot), ~41 issue slots per 64 pixels instead of 2 x 33.  Every pixel still sees the scalar operations in
// the same order with the same roundings.  On the C3 frame the 8x8 patches take 6.77 M hit evaluations and 0.86 M
// segment walks where 8x4 patches of one pixel per lane took 9.98 M and 1.62 M (tests/tools/blend_model.py).
// Other differences that do not change results: colour is staged with the batch instead of fetched from global memory
// per contributing pair (shader.cpp:268-269); the alpha >= 1/255 test is a compare against a per-Gaussian power
// threshold, so no exp is needed to reject; the tile stops as soon as every pixel has saturated (the reference keeps
// loading and barrier-ing until the list ends, shader.cpp:226-277).
//
// Compute-bound (FP32 issue + shared memory), not HBM-bound; HBM side is 4 B id + 48 B record per
// instance (mostly L2 hits) + 12 B per pixel.
#include "blend_walk.cuh"

namespace lcgs_b200 {

// ---- tile schedule: longest list first -----------------------------------------------------------
// Tile populations are heavy-tailed (a tile in front of the object holds ten times the average list), and
// the hardware hands CTAs out in blockIdx order: with tiles in row-major order the kernel's tail is
// whichever long tile happened to start last.  One small CTA buckets the tiles by list length
// (floating-point-like buckets: exponent + 3 mantissa bits, 12 % granularity) and writes the tile ids in
// descending bucket order; blend CTA b then renders tile order[b].  The order inside a bucket is
// whatever the atomics produce -- it changes the schedule only, never a result.
constexpr int kOrderThreads = 1024;
constexpr int kOrderBuckets = 256;

__device__ __forceinline__ uint32_t length_bucket(uint32_t len)
{
    if (len < 8u) return len;  // 0..7 exact
    const int e = 31 - __clz(len);  // >= 3
    return (uint32_t)((e - 2) * 8) + ((len >> (e - 3)) & 7u);  // 8.. : (e-3)*8 + 8 + mantissa
}

__global__ void __launch_bounds__(kOrderThreads)
    tile_order_kernel(const uint2* __restrict__ ranges, uint32_t num_tiles, uint32_t* __restrict__ order,
                      const uint32_t* __restrict__ d_num_rendered, uint32_t capacity, uint32_t* __restrict__ d_flags)
{
    // the frame's capacity check, made where the count lives: [0] = overflow flag, [1] = the capacity it was
    // tested against; both travel back to the host with the count (lcgs_b200_num_rendered)
    if (d_flags && threadIdx.x == 0) {
        d_flags[0] = *d_num_rendered > capacity ? 1u : 0u;
        d_flags[1] = capacity;
    }
    __shared__ uint32_t s_cnt[kOrderBuckets], s_base[kOrderBuckets];
    const int tid = threadIdx.x;
    if (tid < kOrderBuckets) s_cnt[tid] = 0u;
    __syncthreads();
    for (uint32_t t = tid; t < num_tiles; t += kOrderThreads) {
        const uint2 r = __ldg(ranges + t);
        atomicAdd(&s_cnt[length_bucket(r.y > r.x ? r.y - r.x : 0u)], 1u);
    }
    __syncthreads();
    // descending exclusive scan over the 256 buckets by one warp (8 buckets per lane)
    if (tid < 32) {
        uint32_t c[8], sum = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            c[k] = s_cnt[kOrderBuckets - 1 - (tid * 8 + k)];
            sum += c[k];
        }
        uint32_t x = sum;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
            if (tid >= d) x += y;
        }
        uint32_t run = x - sum;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            s_base[kOrderBuckets - 1 - (tid * 8 + k)] = run;
            run += c[k];
        }
    }
    __syncthreads();
    for (uint32_t t = tid; t < num_tiles; t += kOrderThreads) {
        const uint2 r = __ldg(ranges + t);
        order[atomicAdd(&s_base[length_bucket(r.y > r.x ? r.y - r.x : 0u)], 1u)] = t;
    }
}
// AUX (blend2_aux_kernel): the same walk also accumulates the per-pixel outputs of the frame's optional aux planes --
// final alpha 1 - T, depth sum(w_i * z_i) and the number of blended pairs n.  The candidate's view depth z = depth[id]
// is staged with its record by a fourth, 4-byte cp.async into s_z; the record planes are unchanged.  The colour
// arithmetic is the same operations in the same order, so the image is bit-identical with AUX on or off.
template <bool AUX>
__device__ __forceinline__ void blend2_body(const int tid, int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                                            const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                                            const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                                            const uint32_t* __restrict__ d_num_rendered, float* __restrict__ img,
                                            uint8_t* __restrict__ rgb8, const float* __restrict__ depth,
                                            float* __restrict__ out_alpha, float* __restrict__ out_depth,
                                            uint32_t* __restrict__ out_n)
{
    __shared__ float4   s_rec[2][3][kWalkThreads];  // [buffer][plane][slot], planes as in the record (common.cuh)
    __shared__ uint32_t s_cnt[2][kWalkWarps];
    __shared__ float    s_z[2][AUX ? kWalkThreads : 1];  // [buffer][slot]: view depth of the candidate (AUX only)
    const uint32_t zbase = AUX ? (uint32_t)__cvta_generic_to_shared(&s_z[0][0]) : 0u;

    const TilePixels p    = tile_pixels(tid & 31, tid >> 5, order, gx, row0);
    const bool       in_a = p.px < W && p.pya < H, in_b = p.px < W && p.pyb < H;
    const float      pxf  = (float)p.px;                          // no half-pixel offset (Q2)
    const f32x2      npy2 = pack2(-(float)p.pya, -(float)p.pyb);  // my - py == my + (-py), exactly

    // Q10 (whole frames only, see blend2_kernel): blend2_kernel returns before it gets here
    if (AUX && d_num_rendered && *d_num_rendered == 0u) {
        // Q10 leaves the image of an empty frame untouched; the aux planes have no reference counterpart and are
        // cleared, so that they never hold a stale frame
        const size_t pa = (size_t)p.px + (size_t)W * (size_t)p.pya, pb = (size_t)p.px + (size_t)W * (size_t)p.pyb;
        if (in_a) {
            if (out_alpha) out_alpha[pa] = 0.0f;
            if (out_depth) out_depth[pa] = 0.0f;
            if (out_n) out_n[pa] = 0u;
        }
        if (in_b) {
            if (out_alpha) out_alpha[pb] = 0.0f;
            if (out_depth) out_depth[pb] = 0.0f;
            if (out_n) out_n[pb] = 0u;
        }
        return;
    }

    // T < 0 marks a finished pixel (saturated, or outside the image); |T| is its final transmittance.
    // A finished pixel needs no flag in the evaluation: T * (1 - alpha) is negative, so it never blends.
    float Ta = in_a ? 1.0f : -1.0f, Tb = in_b ? 1.0f : -1.0f;
    float c0a = 0.0f, c0b = 0.0f, c1a = 0.0f, c1b = 0.0f, c2a = 0.0f, c2b = 0.0f;
    float    da_sum = 0.0f, db_sum = 0.0f;  // AUX: sum of w * z
    uint32_t na = 0u, nb = 0u;              // AUX: blended pairs
    struct Consts {
        f32x2 one2, l2e2;  // (1, 1), (log2 e, log2 e)
    };
    auto make_consts = [] { return Consts{ bcast2(1.0f), bcast2(1.4426950408889634f) }; };

    auto stage_depth = [&](uint32_t entry, uint32_t id) {
        if constexpr (AUX) cp_async_4(zbase + entry * 4u, depth + id);
    };
    // one Gaussian on this lane's two pixels; blend_power(a, b, c, dx, dy) = fma(b*dx, dy, fma(a*dx, dx, (c*dy)*dy)),
    // dx is shared by the pair
    // (requesting the next hit's geometry planes before evaluating the current one -- two register sets, loop unrolled
    // by two -- measured slower: 0.477 ms at 66 registers / 7 CTAs, 0.533 ms at 64 / 8 against 0.423 ms; packing the
    // cull's survivors densely across the four warps walks a third fewer segments but measured 0.430 ms against 0.423:
    // profiles/README.md)
    auto evaluate = [&](const Consts& k, const float4& ea, const float4& eb, const float4& ec, uint32_t entry) {
        const uint32_t zaddr = zbase + entry * 4u;  // AUX: the entry's staged view depth
        const float    dx   = ea.x - pxf;
        const float adx  = ea.z * dx, bdx = ea.w * dx;
        const f32x2 dy2  = add2(bcast2(ea.y), npy2);
        const f32x2 cdy2 = mul2(bcast2(eb.x), dy2);
        const f32x2 in2  = fma2(bcast2(adx), bcast2(dx), mul2(cdy2, dy2));
        const f32x2 pw2  = fma2(bcast2(bdx), dy2, in2);
        float pwa, pwb;
        unpack2(pw2, pwa, pwb);
        const bool oka = !(pwa > 0.0f) && !(pwa < eb.y);  // shader.cpp:257,259: skipped pairs are predicated off
        const bool okb = !(pwb > 0.0f) && !(pwb < eb.y);
        // alpha = min(0.99, opacity * exp(power)) = min(0.99, 2^(power * log2(e) + log2(opacity)))
        float xa, xb;
        unpack2(fma2(pw2, k.l2e2, bcast2(eb.z)), xa, xb);
        const float alpa = fminf(0.99f, ex2_ftz(xa)), alpb = fminf(0.99f, ex2_ftz(xb));
        const f32x2 al2  = pack2(alpa, alpb);
        const f32x2 T2   = pack2(Ta, Tb);
        float tta, ttb, wa, wb;
        unpack2(mul2(T2, sub2(k.one2, al2)), tta, ttb);  // T * (1 - alpha): < 0 for a finished pixel
        unpack2(mul2(T2, al2), wa, wb);
        const bool bla = oka && !(tta < 0.0001f), blb = okb && !(ttb < 0.0001f);  // shader.cpp:261-265
        const float wsa = bla ? wa : 0.0f, wsb = blb ? wb : 0.0f;
        fma2_acc_s(c0a, c0b, wsa, wsb, ec.x);
        fma2_acc_s(c1a, c1b, wsa, wsb, ec.y);
        fma2_acc_s(c2a, c2b, wsa, wsb, ec.z);
        if constexpr (AUX) {
            fma2_acc_s(da_sum, db_sum, wsa, wsb, lds32(zaddr));
            na += bla;
            nb += blb;
        }
        // saturated (ok but not blended): this entry is dropped and the pixel is finished
        Ta = oka ? (bla ? tta : -fabsf(Ta)) : Ta;
        Tb = okb ? (blb ? ttb : -fabsf(Tb)) : Tb;
    };
    walk_tile(tid, p, ranges, point_list, records, s_rec, s_cnt, Ta, Tb, stage_depth, make_consts, evaluate);

    Ta = fabsf(Ta);
    Tb = fabsf(Tb);
    const float va0 = __fmaf_rn(bg0, Ta, c0a), va1 = __fmaf_rn(bg1, Ta, c1a), va2 = __fmaf_rn(bg2, Ta, c2a);
    const float vb0 = __fmaf_rn(bg0, Tb, c0b), vb1 = __fmaf_rn(bg1, Tb, c1b), vb2 = __fmaf_rn(bg2, Tb, c2b);
    const size_t plane = (size_t)W * (size_t)H;
    if (in_a) {
        const size_t pix = (size_t)p.px + (size_t)W * (size_t)p.pya;
        img[pix] = va0; img[pix + plane] = va1; img[pix + 2 * plane] = va2;
    }
    if (in_b) {
        const size_t pix = (size_t)p.px + (size_t)W * (size_t)p.pyb;
        img[pix] = vb0; img[pix + plane] = vb1; img[pix + 2 * plane] = vb2;
    }
    if constexpr (AUX) {
        const size_t pa = (size_t)p.px + (size_t)W * (size_t)p.pya, pb = (size_t)p.px + (size_t)W * (size_t)p.pyb;
        if (in_a) {
            if (out_alpha) out_alpha[pa] = 1.0f - Ta;
            if (out_depth) out_depth[pa] = da_sum;
            if (out_n) out_n[pa] = na;
        }
        if (in_b) {
            if (out_alpha) out_alpha[pb] = 1.0f - Tb;
            if (out_depth) out_depth[pb] = db_sum;
            if (out_n) out_n[pb] = nb;
        }
    }
    if (rgb8) {
        // The app's post-process fused into the epilogue (app/main.cpp:322-337): HWC, vertical flip, uint8(v * 255) with
        // truncation (cvt.rzi saturates at 0; 255 caps what C leaves undefined).  The tile's 16 x 48 bytes are staged in
        // shared memory (the record buffers are free now) and leave as runs of 32 consecutive bytes per warp instruction:
        // per-pixel byte stores were 96 partial-sector writes per tile, which is what the NVLink ingress of the rank that
        // owns a multi-GPU frame ring chokes on when 7 peers blend into it.
        unsigned char* const s_u8 = reinterpret_cast<unsigned char*>(&s_rec[0][0][0]);
        __syncthreads();  // every warp has left the round loop: nobody reads the record buffers any more
        auto u8 = [](float v) { return (unsigned char)min(__float2uint_rz(v * 255.0f), 255u); };
        if (in_a) {
            const int o = ((p.pya - p.tile_y0) * 16 + (p.px - p.tile_x0)) * 3;
            s_u8[o] = u8(va0); s_u8[o + 1] = u8(va1); s_u8[o + 2] = u8(va2);
        }
        if (in_b) {
            const int o = ((p.pyb - p.tile_y0) * 16 + (p.px - p.tile_x0)) * 3;
            s_u8[o] = u8(vb0); s_u8[o + 1] = u8(vb1); s_u8[o + 2] = u8(vb2);
        }
        __syncthreads();
        const int cols = min(16, W - p.tile_x0) * 3;  // valid bytes per tile row
#pragma unroll
        for (int k = tid; k < 16 * 48; k += kWalkThreads) {
            const int row = k / 48, col = k - row * 48, y = p.tile_y0 + row;
            if (y < H && col < cols) rgb8[((size_t)(H - 1 - y) * (size_t)W + (size_t)p.tile_x0) * 3 + col] = s_u8[k];
        }
    }
}

template <int MIN_CTAS>
__global__ void __launch_bounds__(kWalkThreads, MIN_CTAS)
    blend2_kernel(int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                  const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                  const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                  const uint32_t* __restrict__ d_num_rendered /* non-null: apply quirk Q10 */, float* __restrict__ img,
                  uint8_t* __restrict__ rgb8)
{
    // num_rendered == 0: the reference returns before launching the render and leaves the image untouched
    // (lcgs/src/gs_tile_splatter/impl.cpp:109, quirk Q10).  Only a whole frame does that: the launcher passes no count
    // for a band of tile rows, whose own instance count says nothing about the frame's, so a band always writes bg * T
    // to its tiles.
    if (d_num_rendered && *d_num_rendered == 0u) return;
    blend2_body<false>((int)threadIdx.x, W, H, gx, row0, bg0, bg1, bg2, ranges, order, point_list, records, d_num_rendered,
                       img, rgb8, nullptr, nullptr, nullptr, nullptr);
}

// blend2_kernel plus the aux planes (see blend2_body); each plane pointer may be null on its own.
// depth: the frame's per-Gaussian view depth [P], indexed like the records.
template <int MIN_CTAS>
__global__ void __launch_bounds__(kWalkThreads, MIN_CTAS)
    blend2_aux_kernel(int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                      const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                      const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                      const uint32_t* __restrict__ d_num_rendered /* non-null: apply quirk Q10 */, float* __restrict__ img,
                      uint8_t* __restrict__ rgb8, const float* __restrict__ depth, float* __restrict__ out_alpha,
                      float* __restrict__ out_depth, uint32_t* __restrict__ out_n)
{
    blend2_body<true>((int)threadIdx.x, W, H, gx, row0, bg0, bg1, bg2, ranges, order, point_list, records, d_num_rendered, img,
                      rgb8, depth, out_alpha, out_depth, out_n);
}

// Display::_transpose_shader (app/display.cpp:30-39): planar CHW float -> RGBA8 unorm framebuffer, no flip.
__global__ void __launch_bounds__(256) transpose_rgba8_kernel(int n, const float* __restrict__ img, uchar4* __restrict__ rgba)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= n) return;
    auto unorm = [](float v) { return (unsigned char)__float2uint_rn(fminf(fmaxf(v, 0.0f), 1.0f) * 255.0f); };
    rgba[p] = make_uchar4(unorm(__ldg(img + p)), unorm(__ldg(img + n + p)), unorm(__ldg(img + 2 * (size_t)n + p)), 255);
}

int launch_tile_order(lcgs_b200_ctx* ctx, const uint32_t* ranges, int num_tiles, const uint32_t* d_num_rendered,
                      size_t list_capacity, cudaStream_t s)
{
    if (num_tiles <= 0) return LCGS_B200_OK;
    int rc = ws_reserve(ctx, ctx->tile_order_ws, (size_t)num_tiles * sizeof(uint32_t));
    if (rc) return rc;
    const uint32_t cap = (uint32_t)(list_capacity > 0xFFFFFFFFull ? 0xFFFFFFFFull : list_capacity);
    tile_order_kernel<<<1, kOrderThreads, 0, s>>>(reinterpret_cast<const uint2*>(ranges), (uint32_t)num_tiles,
                                                  (uint32_t*)ctx->tile_order_ws.ptr, d_num_rendered, cap,
                                                  d_num_rendered ? ctx->d_scalars + LCGS_SCALAR_OVERFLOW : nullptr);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

// `ranges` must have been ordered by launch_tile_order on the same stream.
int launch_blend(lcgs_b200_ctx* ctx, int W, int H, const float* bg, const uint32_t* ranges, const uint32_t* point_list,
                 const float4* records, const uint32_t* d_num_rendered, float* img, uint8_t* rgb8, int row0, int row1,
                 cudaStream_t s, const float* depth, float* out_alpha, float* out_depth, uint32_t* out_n)
{
    const uint32_t gx = (uint32_t)((W + 15) / 16), gy = (uint32_t)((H + 15) / 16);
    if (row1 < 0) row1 = (int)gy;
    if (W <= 0 || H <= 0 || row1 <= row0) return LCGS_B200_OK;
    const uint32_t num_tiles = gx * (uint32_t)(row1 - row0);
    // Q10 applies to a whole frame only (see the kernel)
    const bool whole = row0 == 0 && row1 == (int)gy;
    const uint2*    rg  = reinterpret_cast<const uint2*>(ranges);
    const uint32_t* ord = (const uint32_t*)ctx->tile_order_ws.ptr;
    const uint32_t* q10 = whole ? d_num_rendered : nullptr;
    // 44 registers at a launch bound of 10 CTAs per SM.  Measured on the C3 frame (blend stage, ms; NVIDIA B200, power
    // limit not recorded): this kernel at 8 / 9 / 10 / 11 / 12 CTAs per SM 0.408 / 0.409 / 0.407 / 0.429 / 0.429 (11, 12
    // spill).  The geometries it replaced (profiles/README.md): records staged through registers 0.416; that plus a cull
    // against the whole tile 0.420 at best; rounds of 256 0.486 at best; one pixel per lane on 8x4 patches 0.578.
    if (out_alpha || out_depth || out_n) {
        // plus the aux planes: 56 registers at a launch bound of 9 CTAs per SM (at 10 the four extra accumulators spill)
        blend2_aux_kernel<9><<<num_tiles, kWalkThreads, 0, s>>>(W, H, gx, (uint32_t)row0, bg[0], bg[1], bg[2], rg, ord,
                                                                point_list, records, q10, img, rgb8, depth, out_alpha,
                                                                out_depth, out_n);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
        return LCGS_B200_OK;
    }
    blend2_kernel<10><<<num_tiles, kWalkThreads, 0, s>>>(W, H, gx, (uint32_t)row0, bg[0], bg[1], bg[2], rg, ord, point_list,
                                                         records, q10, img, rgb8);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_transpose_rgba8(lcgs_b200_ctx* ctx, int W, int H, const float* img, uint8_t* rgba, cudaStream_t s)
{
    const long n = (long)W * H;
    if (n <= 0) return LCGS_B200_OK;
    transpose_rgba8_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>((int)n, img, reinterpret_cast<uchar4*>(rgba));
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
