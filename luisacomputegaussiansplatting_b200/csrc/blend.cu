// blend.cu -- stage 5b: per-tile front-to-back alpha blending.
// Replaces m_forward_render_shader (lcgs/src/gs_tile_splatter/shader.cpp:171-288).
//
// One 128-thread CTA per 16x16 tile; each warp owns an 8x8 pixel patch, each lane two pixels of it
// (blend2_kernel).  The tile's depth-sorted list is consumed in rounds of 128 candidates through a
// double-buffered shared-memory stage:
//   produce (round r+1): every thread copies one Gaussian's packed 48-byte record (pixel mean,
//      pre-scaled conic, alpha-test threshold, log2 opacity, colour, cull quotients) global -> shared
//      with three 16-byte cp.async (LDGSTS): the record never occupies a register, and the copies land
//      while round r is blended;
//   consume (round r): each warp walks the 4 segments of 32 candidates; per segment one lane per
//      candidate tests it with cull_rect_fast() against the bounding box of the warp's unfinished
//      pixels, and only the ballot's set bits are evaluated, all 64 pixels on the same Gaussian with
//      broadcast LDS.128 and packed FP32 arithmetic.
// There is ONE __syncthreads per round (it also carries the block-wide "every pixel saturated" vote).
// cull_rect_fast() (lcgs_math.cuh; branch-free, its two divisions precomputed per Gaussian in the
// record) is conservative with respect to the per-pixel float evaluation, so culling only removes
// pairs the alpha test would have skipped: on the C3 scene 42 % of the (Gaussian, tile) instances
// binned by the reference's loose rect never touch their tile -- the reference evaluates all of them
// for 256 pixels.  (MODE 0 / 1 of the kernel, tuning library only: the earlier produce step that
// gathered through registers and culled against the whole tile first -- it never saved a segment walk,
// because survivors were compacted per warp.)
// Other differences that do not change results: colour is staged with the batch instead of fetched
// from global memory per contributing pair (shader.cpp:268-269); the alpha >= 1/255 test is a
// compare against a per-Gaussian power threshold, so no exp is needed to reject; the tile stops as
// soon as every pixel has saturated (the reference keeps loading and barrier-ing until the list
// ends, shader.cpp:226-277).
// blend_kernel (one pixel per lane, 8 warps x 8x4 patches) is the kernel blend2_kernel replaced; it is
// compiled into the -DLCGS_TUNING library only, for A/B runs.
//
// Compute-bound (FP32 issue + shared memory), not HBM-bound; HBM side is 4 B id + 48 B record per
// instance (mostly L2 hits) + 12 B per pixel.
#include "common.cuh"

namespace lcgs_b200 {

#ifdef LCGS_TUNING
constexpr int kBlendThreads = 256;
constexpr int kBlendWarps   = kBlendThreads / 32;
#endif

__device__ __forceinline__ float4 lds128(uint32_t addr)
{
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}

__device__ __forceinline__ float lds32(uint32_t addr)
{
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
    return v;
}

__device__ __forceinline__ void sts128(uint32_t addr, const float4& v)
{
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float ex2_ftz(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

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

#ifdef LCGS_TUNING  // the one-pixel-per-lane kernel blend2_kernel replaced; built into the tuning library only, for A/B runs
template <int MIN_CTAS>
__global__ void __launch_bounds__(kBlendThreads, MIN_CTAS)
    blend_kernel(int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                 const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                 const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                 const uint32_t* __restrict__ d_num_rendered /* non-null: apply quirk Q10 */, float* __restrict__ img,
                 uint8_t* __restrict__ rgb8)
{
    // num_rendered == 0: the reference returns before launching the render and leaves the image
    // untouched (lcgs/src/gs_tile_splatter/impl.cpp:109, quirk Q10).  Only a whole frame does that: the
    // launcher passes no count for a band of tile rows, whose own instance count says nothing about the
    // frame's, so a band always writes bg * T to its tiles.
    if (d_num_rendered && *d_num_rendered == 0u) return;

    // [buffer][plane][slot]: plane 0 = (pix.x, pix.y, -0.5*conic.x, -conic.y),
    // plane 1 = (-0.5*conic.z, threshold, log2(opacity), ry), plane 2 = (r, g, b, rx)
    __shared__ float4   s_rec[2][3][kBlendThreads];
    __shared__ uint32_t s_cnt[2][kBlendWarps];

    const int      tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned FULL    = 0xFFFFFFFFu;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t sbase   = (uint32_t)__cvta_generic_to_shared(&s_rec[0][0][0]);
    constexpr uint32_t kPlane = kBlendThreads * 16u, kBuf = 3u * kPlane;

    // 8x4 pixel patch per warp: warps tile the 16x16 block as 2 columns x 4 rows of patches
    const uint32_t tile    = __ldg(order + blockIdx.x);  // band-local tile id, longest lists first
    const uint32_t tile_by = tile / gx, tile_bx = tile - tile_by * gx;
    const int tile_x0 = (int)tile_bx * 16, tile_y0 = (int)(row0 + tile_by) * 16;
    const int patch_x0 = tile_x0 + (warp & 1) * 8, patch_y0 = tile_y0 + (warp >> 1) * 4;
    const int px = patch_x0 + (lane & 7);
    const int py = patch_y0 + (lane >> 3);
    const bool  inside = px < W && py < H;
    const float pxf = (float)px, pyf = (float)py;  // no half-pixel offset (Q2)
    const float tx0 = (float)tile_x0, ty0 = (float)tile_y0, tx1 = (float)(tile_x0 + 15), ty1 = (float)(tile_y0 + 15);

    const uint2    range = __ldg(ranges + tile);
    const uint32_t len   = range.y > range.x ? range.y - range.x : 0u;
    const uint32_t nrounds = (len + kBlendThreads - 1) / kBlendThreads;

    // T < 0 marks a finished pixel (saturated, or outside the image); |T| is its final transmittance.
    // A finished pixel needs no flag in the inner loop: T * (1 - alpha) is negative, so it never blends.
    float T = inside ? 1.0f : -1.0f, C0 = 0.0f, C1 = 0.0f, C2 = 0.0f;

    // cull one gathered candidate against the tile and append it to this warp's segment of `buf`
    auto produce = [&](uint32_t buf, bool valid, const float4& a, const float4& b, const float4& c) {
        const bool     keep = valid && !cull_rect_fast(a.x, a.y, a.z, a.w, b.x, b.y, b.w, c.w, tx0, ty0, tx1, ty1);
        const unsigned kept = __ballot_sync(FULL, keep);
        if (keep) {
            // a warp's survivors fill its segment from the top, earliest candidate in slot 31: the consumer
            // then walks the hit mask from its highest bit, which is a single FLO (no bit reversal)
            const uint32_t slot = warp * 32 + 31 - __popc(kept & lt_mask);
            const uint32_t addr = sbase + buf * kBuf + slot * 16u;
            sts128(addr, a);
            sts128(addr + kPlane, b);
            sts128(addr + 2u * kPlane, c);
        }
        if (lane == 0) s_cnt[buf][warp] = __popc(kept);
    };

    // prologue: round 0 into buffer 0; prefetch the id of round 1
    float4   ra, rb, rc;
    uint32_t next_id = 0;
    {
        const bool valid = (uint32_t)tid < len;
        if (valid) {
            const float4* rec = records + (size_t)__ldg(point_list + range.x + tid) * kRecordFloat4s;
            ra = __ldg(rec); rb = __ldg(rec + 1); rc = __ldg(rec + 2);
        }
        if (kBlendThreads + (uint32_t)tid < len) next_id = __ldg(point_list + range.x + kBlendThreads + tid);
        produce(0u, valid, ra, rb, rc);
    }
    __syncthreads();

    for (uint32_t r = 0; r < nrounds; r++) {
        const uint32_t buf = r & 1u;
        // ---- issue the gathers of round r+1 (consumed after the blend below) ------------------------
        const uint32_t nidx       = (r + 1u) * kBlendThreads + tid;
        const bool     next_valid = nidx < len;
        if (next_valid) {
            const float4* rec = records + (size_t)next_id * kRecordFloat4s;
            ra = __ldg(rec); rb = __ldg(rec + 1); rc = __ldg(rec + 2);
        }
        if (nidx + kBlendThreads < len) next_id = __ldg(point_list + range.x + nidx + kBlendThreads);

        // ---- consume round r: per segment, cull against the patch, evaluate the hits ----------------
        bool done = T < 0.0f;
        if (!__all_sync(FULL, done)) {
            const uint32_t abase = sbase + buf * kBuf;
            // the patch shrinks to the bounding box of the pixels that are still accumulating: saturated
            // pixels need no more Gaussians, so later rounds cull against a smaller rectangle
            const unsigned ax = done ? 255u : (unsigned)(lane & 7), ay = done ? 255u : (unsigned)(lane >> 3);
            const unsigned bx = done ? 0u : (unsigned)(lane & 7), by = done ? 0u : (unsigned)(lane >> 3);
            const float wx0 = (float)(patch_x0 + (int)__reduce_min_sync(FULL, ax));
            const float wy0 = (float)(patch_y0 + (int)__reduce_min_sync(FULL, ay));
            const float wx1 = (float)(patch_x0 + (int)__reduce_max_sync(FULL, bx));
            const float wy1 = (float)(patch_y0 + (int)__reduce_max_sync(FULL, by));
#pragma unroll 1
            for (int seg = 0; seg < kBlendWarps; seg++) {
                const uint32_t cnt     = s_cnt[buf][seg];
                const uint32_t segbase = abase + seg * 512u;
                bool           hit     = false;
                if ((uint32_t)lane + cnt >= 32u) {
                    const float4 ga = lds128(segbase + lane * 16u);
                    const float4 gb = lds128(segbase + kPlane + lane * 16u);
                    const float  rx = lds32(segbase + 2u * kPlane + lane * 16u + 12u);
                    hit             = !cull_rect_fast(ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.w, rx, wx0, wy0, wx1, wy1);
                }
                unsigned hits = __ballot_sync(FULL, hit);
                while (hits) {
                    const int      top  = 31 - __clz(hits);
                    const uint32_t addr = segbase + top * 16u;
                    hits ^= 1u << top;
                    const float4 ea = lds128(addr);
                    const float4 eb = lds128(addr + kPlane);
                    const float4 ec = lds128(addr + 2u * kPlane);
                    // canonical evaluation (shared with the oracle), two explicit fused ops
                    const float power = blend_power(ea.z, ea.w, eb.x, ea.x - pxf, ea.y - pyf);
                    // shader.cpp:257,259: skipped pairs are predicated off
                    const bool  ok     = !(power > 0.0f) && !(power < eb.y);
                    // opacity * exp(power) = 2^(power * log2(e) + log2(opacity)): one FMA in front of MUFU.EX2
                    const float alpha  = fminf(0.99f, ex2_ftz(__fmaf_rn(power, 1.4426950408889634f, eb.z)));
                    const float test_T = T * (1.0f - alpha);         // < 0 for a finished pixel
                    const bool  blend  = ok && !(test_T < 0.0001f);  // shader.cpp:261-265
                    const float w      = blend ? T * alpha : 0.0f;
                    C0 = __fmaf_rn(w, ec.x, C0);
                    C1 = __fmaf_rn(w, ec.y, C1);
                    C2 = __fmaf_rn(w, ec.z, C2);
                    // saturated (ok but not blended): this entry is dropped and the pixel is finished
                    T = ok ? (blend ? test_T : -fabsf(T)) : T;
                }
                done = T < 0.0f;
                if (__all_sync(FULL, done)) break;
            }
        }

        // ---- produce round r+1 into the other buffer ------------------------------------------------
        if (r + 1u < nrounds) produce(buf ^ 1u, next_valid, ra, rb, rc);
        // one barrier per round: publishes buffer buf^1, retires buffer buf, votes on early exit
        if (__syncthreads_and(T < 0.0f)) break;
    }

    T = fabsf(T);
    const float v0 = __fmaf_rn(bg0, T, C0), v1 = __fmaf_rn(bg1, T, C1), v2 = __fmaf_rn(bg2, T, C2);
    if (inside) {
        const size_t plane = (size_t)W * (size_t)H;
        const size_t pix   = (size_t)px + (size_t)W * (size_t)py;
        img[pix]             = v0;
        img[pix + plane]     = v1;
        img[pix + 2 * plane] = v2;
    }
    if (rgb8) {
        // The app's post-process fused into the epilogue (app/main.cpp:322-337): HWC, vertical flip, uint8(v * 255) with
        // truncation (cvt.rzi saturates at 0; 255 caps what C leaves undefined).  The tile's 16 x 48 bytes are staged in
        // shared memory (the record buffers are free now) and leave as runs of 32 consecutive bytes per warp instruction:
        // per-pixel byte stores were 96 partial-sector writes per tile, which is what the NVLink ingress of the rank that
        // owns a multi-GPU frame ring chokes on when 7 peers blend into it.
        unsigned char* const s_u8 = reinterpret_cast<unsigned char*>(&s_rec[0][0][0]);
        __syncthreads();  // every warp has left the round loop: nobody reads the record buffers any more
        if (inside) {
            const int o = ((py - tile_y0) * 16 + (px - tile_x0)) * 3;
            s_u8[o]     = (unsigned char)min(__float2uint_rz(v0 * 255.0f), 255u);
            s_u8[o + 1] = (unsigned char)min(__float2uint_rz(v1 * 255.0f), 255u);
            s_u8[o + 2] = (unsigned char)min(__float2uint_rz(v2 * 255.0f), 255u);
        }
        __syncthreads();
        const int cols = min(16, W - tile_x0) * 3;  // valid bytes per tile row
#pragma unroll
        for (int k = tid; k < 16 * 48; k += kBlendThreads) {
            const int row = k / 48, col = k - row * 48, y = tile_y0 + row;
            if (y < H && col < cols) rgb8[((size_t)(H - 1 - y) * (size_t)W + (size_t)tile_x0) * 3 + col] = s_u8[k];
        }
    }
}

#endif  // LCGS_TUNING

// ---- two pixels per lane: 8x8 patches, packed FP32 ------------------------------------------------
// Same algorithm, other shape: four warps per tile, each owning an 8x8 patch, lane = pixels (x, y) and
// (x, y + 4).  A Gaussian that hits the patch is fetched once for 64 pixels, and the per-pixel arithmetic
// of the pair runs on Blackwell's packed FP32 instructions (FADD2 / FMUL2 / FFMA2: two IEEE binary32
// operations per lane and issue slot, per-Gaussian operands broadcast with the .F32 operand form), so the
// inner loop is ~41 issue slots per 64 pixels instead of 2 x 33.  On the C3 frame the 8x8 patches take
// 6.77 M hit evaluations and 0.86 M segment walks where the 8x4 patches take 9.98 M and 1.62 M
// (tests/tools/blend_model.py replays both schedules on the oracle frame).  Every pixel still sees the same
// operations in the same order with the same roundings, so the image is bit-identical to blend_kernel's.
constexpr int kB2Threads = 128;
constexpr int kB2Warps   = kB2Threads / 32;

typedef unsigned long long f32x2;

__device__ __forceinline__ f32x2 pack2(float lo, float hi)
{
    f32x2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi)
{
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 bcast2(float x) { return pack2(x, x); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b)
{
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c)
{
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// acc = a * b + acc in place (one register pair for the loop-carried accumulator: no copies)
__device__ __forceinline__ void fma2_acc(f32x2& acc, f32x2 a, f32x2 b)
{
    asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
// (ca, cb) += (wa, wb) * e, the accumulators living in two scalar registers
__device__ __forceinline__ void fma2_acc_s(float& ca, float& cb, float wa, float wb, float e)
{
    asm("{\n\t.reg .b64 c, w, x;\n\tmov.b64 c, {%0, %1};\n\tmov.b64 w, {%2, %3};\n\tmov.b64 x, {%4, %4};\n\t"
        "fma.rn.f32x2 c, w, x, c;\n\tmov.b64 {%0, %1}, c;\n\t}"
        : "+f"(ca), "+f"(cb)
        : "f"(wa), "f"(wb), "f"(e));
}
// 1 << pos without a constant register (BMSK)
__device__ __forceinline__ unsigned bit_at(int pos)
{
    unsigned r;
    asm("bmsk.clamp.b32 %0, %1, 1;" : "=r"(r) : "r"(pos));
    return r;
}
// 16-byte asynchronous copy global -> shared (LDGSTS.128): the data never occupies a register
__device__ __forceinline__ void cp_async_16(uint32_t smem_addr, const void* gptr)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_4(uint32_t smem_addr, const void* gptr)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all2() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }
// index of the highest set bit (FLO), x != 0
__device__ __forceinline__ int top_bit(unsigned x)
{
    int r;
    asm("bfind.u32 %0, %1;" : "=r"(r) : "r"(x));
    return r;
}

// CPT = candidates per thread and round (1 or 2): rounds of 128 * CPT list entries, 4 * CPT segments
// MODE 0: the produce step culls each gathered candidate against the whole tile and compacts the survivors per warp.
// MODE 1: no tile cull -- survivors are compacted per warp, not across warps, so the tile cull never removes a segment
//         walk, and whatever it removes the patch cull removes too (a candidate it would have dropped costs one lane of
//         a patch cull that runs anyway).
// MODE 2 (CPT = 1): as MODE 1, and the records never pass through registers: each thread copies its candidate's three
//         16-byte planes global -> shared with cp.async (LDGSTS) straight into its slot of the next round's buffer,
//         waited for before the round's barrier.
//
// AUX (blend2_aux_kernel, MODE 2 only): the same walk also accumulates the per-pixel outputs of the frame's optional
// aux planes -- final alpha 1 - T, depth sum(w_i * z_i) and the number of blended pairs n.  The candidate's view depth
// z = depth[id] is staged with its record by a fourth, 4-byte cp.async into s_z; the record planes are unchanged.  The
// colour arithmetic is the same operations in the same order, so the image is bit-identical with AUX on or off.
// `tid` is threadIdx.x read in the __global__ wrapper: there the compiler knows it is below the launch bound (128) and
// folds the index arithmetic as it did when this was the kernel's own body; read here, it would not.
template <int MIN_CTAS, int CPT, int MODE, bool AUX>
__device__ __forceinline__ void blend2_body(const int tid, int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                                            const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                                            const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                                            const uint32_t* __restrict__ d_num_rendered, float* __restrict__ img,
                                            uint8_t* __restrict__ rgb8, const float* __restrict__ depth,
                                            float* __restrict__ out_alpha, float* __restrict__ out_depth,
                                            uint32_t* __restrict__ out_n)
{
    static_assert(!AUX || (MODE == 2 && CPT == 1), "the aux outputs are written for the asynchronous staging only");

    constexpr int kB2Round = kB2Threads * CPT, kB2Segs = kB2Round / 32;
    __shared__ float4   s_rec[2][3][kB2Round];  // [buffer][plane][slot], planes as in blend_kernel
    __shared__ uint32_t s_cnt[2][kB2Segs];
    __shared__ float    s_z[2][AUX ? kB2Round : 1];  // [buffer][slot]: view depth of the candidate (AUX only)

    const int      lane = tid & 31, warp = tid >> 5;
    const unsigned FULL    = 0xFFFFFFFFu;
    const unsigned lt_mask = (1u << lane) - 1u;
    const uint32_t sbase   = (uint32_t)__cvta_generic_to_shared(&s_rec[0][0][0]);
    constexpr uint32_t kPlane = kB2Round * 16u, kBuf = 3u * kPlane;
    const uint32_t zbase = AUX ? (uint32_t)__cvta_generic_to_shared(&s_z[0][0]) : 0u;

    const uint32_t tile    = __ldg(order + blockIdx.x);  // band-local tile id, longest lists first
    const uint32_t tile_by = tile / gx, tile_bx = tile - tile_by * gx;
    const int tile_x0 = (int)tile_bx * 16, tile_y0 = (int)(row0 + tile_by) * 16;
    const int patch_x0 = tile_x0 + (warp & 1) * 8, patch_y0 = tile_y0 + (warp >> 1) * 8;
    const int px = patch_x0 + (lane & 7);
    const int pya = patch_y0 + (lane >> 3), pyb = pya + 4;
    const bool  in_a = px < W && pya < H, in_b = px < W && pyb < H;
    const float pxf  = (float)px;                                  // no half-pixel offset (Q2)
    const f32x2 npy2 = pack2(-(float)pya, -(float)pyb);            // my - py == my + (-py), exactly
    const float tx0 = (float)tile_x0, ty0 = (float)tile_y0, tx1 = (float)(tile_x0 + 15), ty1 = (float)(tile_y0 + 15);

    // Q10 (whole frames only, see blend_kernel): blend2_kernel returns before it gets here
    if (AUX && d_num_rendered && *d_num_rendered == 0u) {
        // Q10 leaves the image of an empty frame untouched; the aux planes have no reference counterpart and are
        // cleared, so that they never hold a stale frame
        const size_t pa = (size_t)px + (size_t)W * (size_t)pya, pb = (size_t)px + (size_t)W * (size_t)pyb;
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

    const uint2    range = __ldg(ranges + tile);
    const uint32_t len   = range.y > range.x ? range.y - range.x : 0u;
    const uint32_t nrounds = (len + kB2Round - 1) / kB2Round;

    // T < 0 marks a finished pixel, as in blend_kernel
    float Ta = in_a ? 1.0f : -1.0f, Tb = in_b ? 1.0f : -1.0f;
    float c0a = 0.0f, c0b = 0.0f, c1a = 0.0f, c1b = 0.0f, c2a = 0.0f, c2b = 0.0f;
    float    da_sum = 0.0f, db_sum = 0.0f;  // AUX: sum of w * z
    uint32_t na = 0u, nb = 0u;              // AUX: blended pairs

    // candidate j (0, 1) of a thread is entry j * 128 + tid of the round: warp w's j-th ballot fills segment j * 4 + w,
    // so segment s holds entries [32 s, 32 s + 32) and the consumers meet the list in order
    auto produce = [&](uint32_t buf, int j, bool valid, const float4& a, const float4& b, const float4& c) {
        const bool     keep = valid && (MODE != 0 || !cull_rect_fast(a.x, a.y, a.z, a.w, b.x, b.y, b.w, c.w, tx0, ty0, tx1, ty1));
        const unsigned kept = __ballot_sync(FULL, keep);
        const uint32_t seg  = (uint32_t)(j * kB2Warps + warp);
        if (keep) {
            const uint32_t slot = seg * 32 + 31 - __popc(kept & lt_mask);  // filled from the top (FLO walk)
            const uint32_t addr = sbase + buf * kBuf + slot * 16u;
            sts128(addr, a);
            sts128(addr + kPlane, b);
            sts128(addr + 2u * kPlane, c);
        }
        if (lane == 0) s_cnt[buf][seg] = __popc(kept);
    };

    // MODE 2: entry `lane` of the warp's 32 candidates goes to slot 31 - lane of the warp's segment (filled from the top)
    auto stage_async = [&](uint32_t buf, bool valid, uint32_t id) {
        if (valid) {
            const float4*  rec  = records + (size_t)id * kRecordFloat4s;
            const uint32_t addr = sbase + buf * kBuf + (uint32_t)(warp * 32 + 31 - lane) * 16u;
            cp_async_16(addr, rec);  // .ca: with .cg (L1 bypass) the blend measured 0.4215 against 0.412 ms
            cp_async_16(addr + kPlane, rec + 1);
            cp_async_16(addr + 2u * kPlane, rec + 2);
            if constexpr (AUX) cp_async_4(zbase + (buf * kB2Round + (uint32_t)(warp * 32 + 31 - lane)) * 4u, depth + id);
        }
        const unsigned v = __ballot_sync(FULL, valid);
        if (lane == 0) s_cnt[buf][warp] = __popc(v);
    };
    static_assert(MODE != 2 || CPT == 1, "asynchronous staging is written for one candidate per thread");

    float4   ra0, rb0, rc0, ra1, rb1, rc1;
    uint32_t next_id0 = 0, next_id1 = 0;
    if (MODE == 2) {
        const bool v0 = (uint32_t)tid < len;
        stage_async(0u, v0, v0 ? __ldg(point_list + range.x + tid) : 0u);
        if (kB2Round + (uint32_t)tid < len) next_id0 = __ldg(point_list + range.x + kB2Round + tid);
        cp_async_wait_all2();
    } else {
        const bool v0 = (uint32_t)tid < len, v1 = CPT == 2 && (uint32_t)tid + kB2Threads < len;
        if (v0) {
            const float4* rec = records + (size_t)__ldg(point_list + range.x + tid) * kRecordFloat4s;
            ra0 = __ldg(rec); rb0 = __ldg(rec + 1); rc0 = __ldg(rec + 2);
        }
        if (v1) {
            const float4* rec = records + (size_t)__ldg(point_list + range.x + kB2Threads + tid) * kRecordFloat4s;
            ra1 = __ldg(rec); rb1 = __ldg(rec + 1); rc1 = __ldg(rec + 2);
        }
        if (kB2Round + (uint32_t)tid < len) next_id0 = __ldg(point_list + range.x + kB2Round + tid);
        if (CPT == 2 && kB2Round + kB2Threads + (uint32_t)tid < len) next_id1 = __ldg(point_list + range.x + kB2Round + kB2Threads + tid);
        produce(0u, 0, v0, ra0, rb0, rc0);
        if (CPT == 2) produce(0u, 1, v1, ra1, rb1, rc1);
    }
    __syncthreads();

    const f32x2 one2 = bcast2(1.0f), l2e2 = bcast2(1.4426950408889634f);

    for (uint32_t r = 0; r < nrounds; r++) {
        const uint32_t buf = r & 1u;
        // ---- issue the gathers of round r+1 ---------------------------------------------------------------
        const uint32_t nidx0 = (r + 1u) * kB2Round + tid, nidx1 = nidx0 + kB2Threads;
        const bool     nv0 = nidx0 < len, nv1 = CPT == 2 && nidx1 < len;
        if (MODE == 2) {
            if (r + 1u < nrounds) stage_async(buf ^ 1u, nv0, next_id0);  // lands while round r is blended
        } else if (nv0) {
            const float4* rec = records + (size_t)next_id0 * kRecordFloat4s;
            ra0 = __ldg(rec); rb0 = __ldg(rec + 1); rc0 = __ldg(rec + 2);
        }
        if (nv1) {
            const float4* rec = records + (size_t)next_id1 * kRecordFloat4s;
            ra1 = __ldg(rec); rb1 = __ldg(rec + 1); rc1 = __ldg(rec + 2);
        }
        if (nidx0 + kB2Round < len) next_id0 = __ldg(point_list + range.x + nidx0 + kB2Round);
        if (CPT == 2 && nidx1 + kB2Round < len) next_id1 = __ldg(point_list + range.x + nidx1 + kB2Round);

        // ---- consume round r -------------------------------------------------------------------------------
        bool da = Ta < 0.0f, db = Tb < 0.0f;
        if (!__all_sync(FULL, da && db)) {
            const uint32_t abase = sbase + buf * kBuf;
            // bounding box of the pixels of the patch that are still accumulating
            const unsigned lx = (unsigned)(lane & 7), ly = (unsigned)(lane >> 3);
            const unsigned ax = (da && db) ? 255u : lx, bx = (da && db) ? 0u : lx;
            const unsigned ay = !da ? ly : (!db ? ly + 4u : 255u), by = !db ? ly + 4u : (!da ? ly : 0u);
            const float wx0 = (float)(patch_x0 + (int)__reduce_min_sync(FULL, ax));
            const float wy0 = (float)(patch_y0 + (int)__reduce_min_sync(FULL, ay));
            const float wx1 = (float)(patch_x0 + (int)__reduce_max_sync(FULL, bx));
            const float wy1 = (float)(patch_y0 + (int)__reduce_max_sync(FULL, by));
#pragma unroll 1
            for (int seg = 0; seg < kB2Segs; seg++) {
                const uint32_t cnt     = s_cnt[buf][seg];
                const uint32_t segbase = abase + seg * 512u;
                bool           hit     = false;
                if ((uint32_t)lane + cnt >= 32u) {
                    const float4 ga = lds128(segbase + lane * 16u);
                    const float4 gb = lds128(segbase + kPlane + lane * 16u);
                    const float  rx = lds32(segbase + 2u * kPlane + lane * 16u + 12u);
                    hit             = !cull_rect_fast(ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.w, rx, wx0, wy0, wx1, wy1);
                }
                unsigned hits = __ballot_sync(FULL, hit);
                // one Gaussian on this lane's two pixels; blend_power(a, b, c, dx, dy) = fma(b*dx, dy, fma(a*dx, dx, (c*dy)*dy)),
                // dx is shared by the pair
                auto evaluate = [&](const float4& ea, const float4& eb, const float4& ec, uint32_t zaddr) {
                    const float dx   = ea.x - pxf;
                    const float adx  = ea.z * dx, bdx = ea.w * dx;
                    const f32x2 dy2  = add2(bcast2(ea.y), npy2);
                    const f32x2 cdy2 = mul2(bcast2(eb.x), dy2);
                    const f32x2 in2  = fma2(bcast2(adx), bcast2(dx), mul2(cdy2, dy2));
                    const f32x2 pw2  = fma2(bcast2(bdx), dy2, in2);
                    float pwa, pwb;
                    unpack2(pw2, pwa, pwb);
                    const bool oka = !(pwa > 0.0f) && !(pwa < eb.y);  // shader.cpp:257,259
                    const bool okb = !(pwb > 0.0f) && !(pwb < eb.y);
                    // alpha = min(0.99, 2^(power * log2(e) + log2(opacity)))
                    float xa, xb;
                    unpack2(fma2(pw2, l2e2, bcast2(eb.z)), xa, xb);
                    const float alpa = fminf(0.99f, ex2_ftz(xa)), alpb = fminf(0.99f, ex2_ftz(xb));
                    const f32x2 al2  = pack2(alpa, alpb);
                    const f32x2 T2   = pack2(Ta, Tb);
                    float tta, ttb, wa, wb;
                    unpack2(mul2(T2, sub2(one2, al2)), tta, ttb);  // T * (1 - alpha): < 0 for a finished pixel
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
                    Ta = oka ? (bla ? tta : -fabsf(Ta)) : Ta;
                    Tb = okb ? (blb ? ttb : -fabsf(Tb)) : Tb;
                };
                // (requesting the next hit's geometry planes before evaluating the current one -- two register sets, loop
                // unrolled by two -- measured slower: 0.477 ms at 66 registers / 7 CTAs, 0.533 ms at 64 / 8 against 0.423 ms;
                // packing the tile cull's survivors densely across the four warps -- counts triple-buffered, cull + count of
                // round r+2 before the barrier of round r, store after it -- walks a third fewer segments but measured
                // 0.430 ms against 0.423: profiles/README.md)
                while (hits) {
                    const int      top  = top_bit(hits);
                    const uint32_t addr = segbase + top * 16u;
                    hits ^= bit_at(top);
                    const float4 ea = lds128(addr);
                    const float4 eb = lds128(addr + kPlane);
                    const float4 ec = lds128(addr + 2u * kPlane);
                    evaluate(ea, eb, ec, zbase + (buf * kB2Round + (uint32_t)seg * 32u + (uint32_t)top) * 4u);
                }
                da = Ta < 0.0f;
                db = Tb < 0.0f;
                if (__all_sync(FULL, da && db)) break;
            }
        }

        // ---- produce round r+1 into the other buffer --------------------------------------------------------
        if (MODE == 2) {
            cp_async_wait_all2();  // this thread's copies have landed; the barrier publishes everybody's
        } else if (r + 1u < nrounds) {
            produce(buf ^ 1u, 0, nv0, ra0, rb0, rc0);
            if (CPT == 2) produce(buf ^ 1u, 1, nv1, ra1, rb1, rc1);
        }
        if (__syncthreads_and(Ta < 0.0f && Tb < 0.0f)) break;
    }

    Ta = fabsf(Ta);
    Tb = fabsf(Tb);
    const float va0 = __fmaf_rn(bg0, Ta, c0a), va1 = __fmaf_rn(bg1, Ta, c1a), va2 = __fmaf_rn(bg2, Ta, c2a);
    const float vb0 = __fmaf_rn(bg0, Tb, c0b), vb1 = __fmaf_rn(bg1, Tb, c1b), vb2 = __fmaf_rn(bg2, Tb, c2b);
    const size_t plane = (size_t)W * (size_t)H;
    if (in_a) {
        const size_t pix = (size_t)px + (size_t)W * (size_t)pya;
        img[pix] = va0; img[pix + plane] = va1; img[pix + 2 * plane] = va2;
    }
    if (in_b) {
        const size_t pix = (size_t)px + (size_t)W * (size_t)pyb;
        img[pix] = vb0; img[pix + plane] = vb1; img[pix + 2 * plane] = vb2;
    }
    if constexpr (AUX) {
        const size_t pa = (size_t)px + (size_t)W * (size_t)pya, pb = (size_t)px + (size_t)W * (size_t)pyb;
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
        // the app's post-process as in blend_kernel: staged in shared memory, 32-byte runs per warp instruction
        unsigned char* const s_u8 = reinterpret_cast<unsigned char*>(&s_rec[0][0][0]);
        __syncthreads();
        auto u8 = [](float v) { return (unsigned char)min(__float2uint_rz(v * 255.0f), 255u); };
        if (in_a) {
            const int o = ((pya - tile_y0) * 16 + (px - tile_x0)) * 3;
            s_u8[o] = u8(va0); s_u8[o + 1] = u8(va1); s_u8[o + 2] = u8(va2);
        }
        if (in_b) {
            const int o = ((pyb - tile_y0) * 16 + (px - tile_x0)) * 3;
            s_u8[o] = u8(vb0); s_u8[o + 1] = u8(vb1); s_u8[o + 2] = u8(vb2);
        }
        __syncthreads();
        const int cols = min(16, W - tile_x0) * 3;
#pragma unroll
        for (int k = tid; k < 16 * 48; k += kB2Threads) {
            const int row = k / 48, col = k - row * 48, y = tile_y0 + row;
            if (y < H && col < cols) rgb8[((size_t)(H - 1 - y) * (size_t)W + (size_t)tile_x0) * 3 + col] = s_u8[k];
        }
    }
}

template <int MIN_CTAS, int CPT, int MODE = 0>
__global__ void __launch_bounds__(kB2Threads, MIN_CTAS)
    blend2_kernel(int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                  const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                  const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                  const uint32_t* __restrict__ d_num_rendered /* non-null: apply quirk Q10 */, float* __restrict__ img,
                  uint8_t* __restrict__ rgb8)
{
    if (d_num_rendered && *d_num_rendered == 0u) return;  // Q10, whole frames only (see blend_kernel)
    blend2_body<MIN_CTAS, CPT, MODE, false>((int)threadIdx.x, W, H, gx, row0, bg0, bg1, bg2, ranges, order, point_list, records, d_num_rendered,
                                            img, rgb8, nullptr, nullptr, nullptr, nullptr);
}

// blend2_kernel<MIN_CTAS, 1, 2> plus the aux planes (see blend2_body); each plane pointer may be null on its own.
// depth: the frame's per-Gaussian view depth [P], indexed like the records.
template <int MIN_CTAS>
__global__ void __launch_bounds__(kB2Threads, MIN_CTAS)
    blend2_aux_kernel(int W, int H, uint32_t gx, uint32_t row0, float bg0, float bg1, float bg2,
                      const uint2* __restrict__ ranges, const uint32_t* __restrict__ order,
                      const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                      const uint32_t* __restrict__ d_num_rendered /* non-null: apply quirk Q10 */, float* __restrict__ img,
                      uint8_t* __restrict__ rgb8, const float* __restrict__ depth, float* __restrict__ out_alpha,
                      float* __restrict__ out_depth, uint32_t* __restrict__ out_n)
{
    blend2_body<MIN_CTAS, 1, 2, true>((int)threadIdx.x, W, H, gx, row0, bg0, bg1, bg2, ranges, order, point_list, records, d_num_rendered, img,
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
    // two pixels per lane, 4 warps per tile, rounds of 128 candidates staged with cp.async, no cull against the whole tile
    // (MODE 2): 44 registers at a launch bound of 10 CTAs per SM.  Measured on the C3 frame (blend stage, ms):
    //   MODE 2 at 8 / 9 / 10 / 11 / 12 CTAs per SM            0.408 / 0.409 / 0.407 / 0.429 / 0.429 (11, 12: spills)
    //   MODE 1 (registers, no tile cull) at 8                  0.416
    //   MODE 0 (registers, tile cull + per-warp compaction)    one candidate per thread at 6 / 7 / 8 / 9 / 10 CTAs per SM
    //                                                          0.451 / 0.432 / 0.420 / 0.439 / 0.463 (10: 48 registers,
    //                                                          spills); two candidates per thread (rounds of 256) at
    //                                                          5 / 6 / 7 / 8: 0.524 / 0.487 / 0.486 / 0.630
    if (out_alpha || out_depth || out_n) {
        // the production geometry plus the aux planes: 56 registers at a launch bound of 9 CTAs per SM (at 10 the four
        // extra accumulators spill)
        blend2_aux_kernel<9><<<num_tiles, kB2Threads, 0, s>>>(W, H, gx, (uint32_t)row0, bg[0], bg[1], bg[2], rg, ord, point_list,
                                                                     records, q10, img, rgb8, depth, out_alpha, out_depth, out_n);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
        return LCGS_B200_OK;
    }
    auto kern2 = blend2_kernel<10, 1, 2>;
#ifdef LCGS_TUNING
    {   // A/B selection (tuning library only): LCGS_BLEND2_MODE 0 / 1 / 2, LCGS_BLEND2_CPT 1 / 2 (mode 0), LCGS_BLEND2_OCC
        const int occ = LCGS_TUNE_INT("LCGS_BLEND2_OCC", 0), cpt = LCGS_TUNE_INT("LCGS_BLEND2_CPT", 1);
        const int mode = LCGS_TUNE_INT("LCGS_BLEND2_MODE", 2);
        if (cpt == 2) {
            kern2 = occ == 5 ? blend2_kernel<5, 2> : occ == 6 ? blend2_kernel<6, 2> : occ == 8 ? blend2_kernel<8, 2> : blend2_kernel<7, 2>;
        } else if (mode == 0) {
            kern2 = occ == 6 ? blend2_kernel<6, 1> : occ == 7 ? blend2_kernel<7, 1> : occ == 9 ? blend2_kernel<9, 1>
                  : occ == 10 ? blend2_kernel<10, 1> : blend2_kernel<8, 1>;
        } else if (mode == 1) {
            kern2 = occ == 7 ? blend2_kernel<7, 1, 1> : occ == 9 ? blend2_kernel<9, 1, 1> : blend2_kernel<8, 1, 1>;
        } else {
            kern2 = occ == 8 ? blend2_kernel<8, 1, 2> : occ == 9 ? blend2_kernel<9, 1, 2> : occ == 11 ? blend2_kernel<11, 1, 2>
                  : occ == 12 ? blend2_kernel<12, 1, 2> : blend2_kernel<10, 1, 2>;
        }
    }
    if (LCGS_TUNE_INT("LCGS_BLEND_P2", 1) == 0) {
        // the one-pixel-per-lane kernel (8x4 patches, 48 registers -> 5 CTAs per SM), kept for A/B runs
        auto      kern = blend_kernel<5>;
        const int occ  = LCGS_TUNE_INT("LCGS_BLEND_OCC", 5);
        if (occ == 4) kern = blend_kernel<4>;
        if (occ == 6) kern = blend_kernel<6>;
        kern<<<num_tiles, kBlendThreads, 0, s>>>(W, H, gx, (uint32_t)row0, bg[0], bg[1], bg[2], rg, ord, point_list, records, q10, img, rgb8);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
        return LCGS_B200_OK;
    }
#endif
    kern2<<<num_tiles, kB2Threads, 0, s>>>(W, H, gx, (uint32_t)row0, bg[0], bg[1], bg[2], rg, ord, point_list, records, q10, img, rgb8);
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
