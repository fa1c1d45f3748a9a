// blend_walk.cuh -- the per-tile front-to-back walk shared by the forward blend (blend.cu) and the blend backward
// (backward.cu), and the PTX helpers both use.
//
// One 128-thread CTA per 16x16 tile; each warp owns an 8x8 pixel patch, each lane the two pixels (x, y) and (x, y + 4)
// of it.  The tile's depth-sorted list is consumed in rounds of 128 candidates through a double-buffered shared-memory
// stage:
//   stage (round r+1): every thread copies one Gaussian's packed 48-byte record (common.cuh) global -> shared with
//      three 16-byte cp.async (LDGSTS), plus an optional per-slot side value chosen by the kernel; the record never
//      occupies a register, and the copies land while round r is walked;
//   walk (round r): each warp walks the 4 segments of 32 candidates; per segment one lane per candidate tests it with
//      cull_rect_fast() against the bounding box of the warp's unfinished pixels, and only the ballot's set bits are
//      handed to the kernel's per-hit callable, highest bit (= earliest entry) first.
// There is ONE __syncthreads per round; it also carries the block-wide "every pixel finished" vote.  cull_rect_fast()
// is conservative with respect to the per-pixel evaluation, so culling only removes pairs the alpha test would have
// skipped, and the forward and the backward, walking with the same code, see every pixel's entries in the same order.
#pragma once
#include "common.cuh"

namespace lcgs_b200 {

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

// 2^x on MUFU.EX2: the blend's alpha is 2^(power * log2(e) + log2(opacity))
__device__ __forceinline__ float ex2_ftz(float x)
{
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// Packed FP32 (FADD2 / FMUL2 / FFMA2): two IEEE binary32 operations per lane and issue slot.
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

constexpr int      kWalkThreads = 128;  // CTA size: four warps, one 8x8 patch each
constexpr int      kWalkWarps   = kWalkThreads / 32;
constexpr uint32_t kWalkPlane   = kWalkThreads * 16u, kWalkBuf = 3u * kWalkPlane;  // bytes of s_rec[.][plane], s_rec[buf]

// The CTA's tile (blend CTA b renders tile order[b], longest lists first) and this lane's two pixels.  Whether a pixel
// lies inside the image is left to the kernel (px < W && py < H), which starts an outside pixel finished (T = -1).
struct TilePixels {
    int      lane, warp;  // tid & 31, tid >> 5
    uint32_t tile;        // band-local tile id
    int      tile_x0, tile_y0, patch_x0, patch_y0;
    int      px, pya, pyb;  // pixels (px, pya) and (px, pyb = pya + 4)
};

__device__ __forceinline__ TilePixels tile_pixels(const int lane, const int warp, const uint32_t* __restrict__ order,
                                                  uint32_t gx, uint32_t row0)
{
    TilePixels p;
    p.lane = lane; p.warp = warp;
    p.tile = __ldg(order + blockIdx.x);
    const uint32_t tile_by = p.tile / gx, tile_bx = p.tile - tile_by * gx;
    p.tile_x0  = (int)tile_bx * 16;
    p.tile_y0  = (int)(row0 + tile_by) * 16;
    p.patch_x0 = p.tile_x0 + (warp & 1) * 8;
    p.patch_y0 = p.tile_y0 + (warp >> 1) * 8;
    p.px       = p.patch_x0 + (lane & 7);
    p.pya      = p.patch_y0 + (lane >> 3);
    p.pyb      = p.pya + 4;
    return p;
}

// Walks the tile's list front to back.  Ta and Tb are the transmittances of the lane's two pixels, updated by `hit`;
// T < 0 marks a finished pixel (saturated, or outside the image), which the cull no longer covers, and the tile stops
// once every pixel has finished.
//   stage_side(entry, id): called when Gaussian `id` is staged into s_rec[entry / 128][.][entry % 128], to stage a
//      per-slot side value of the kernel's own (issued with cp.async, it has landed by the round's barrier).
//   make_consts(): called once, after round 0 has been staged; its result is handed to every hit.  Values the per-hit
//      work keeps in registers are set up here, after the prologue, where the forward blend has always set them up
//      (set up before the walk, they change the forward's schedule).
//   hit(consts, ea, eb, ec, entry): the three record planes of the next entry that passed the cull, in list order.
// lane and warp come from the caller's tid (tile_pixels), and `tid` itself is threadIdx.x read in the __global__
// function: there the compiler knows it is below the launch bound and folds the index arithmetic.
template <typename StageSide, typename MakeConsts, typename Hit>
__device__ __forceinline__ void walk_tile(const int tid, const TilePixels& p, const uint2* __restrict__ ranges,
                                          const uint32_t* __restrict__ point_list, const float4* __restrict__ records,
                                          float4 (&s_rec)[2][3][kWalkThreads], uint32_t (&s_cnt)[2][kWalkWarps],
                                          const float& Ta, const float& Tb, StageSide stage_side, MakeConsts make_consts,
                                          Hit hit)
{
    const int      lane = p.lane, warp = p.warp;
    const unsigned FULL  = 0xFFFFFFFFu;
    const uint32_t sbase = (uint32_t)__cvta_generic_to_shared(&s_rec[0][0][0]);

    const uint2    range   = __ldg(ranges + p.tile);
    const uint32_t len     = range.y > range.x ? range.y - range.x : 0u;
    const uint32_t nrounds = (len + kWalkThreads - 1) / kWalkThreads;

    // entry `lane` of the warp's 32 candidates goes to slot 31 - lane of the warp's segment: filled from the top, the
    // walk from the highest hit bit (one FLO, no bit reversal) meets the list in order
    auto stage = [&](uint32_t buf, bool valid, uint32_t id) {
        if (valid) {
            const float4*  rec  = records + (size_t)id * kRecordFloat4s;
            const uint32_t slot = (uint32_t)(warp * 32 + 31 - lane);
            const uint32_t addr = sbase + buf * kWalkBuf + slot * 16u;
            cp_async_16(addr, rec);  // .ca: with .cg (L1 bypass) the blend measured 0.4215 against 0.412 ms
            cp_async_16(addr + kWalkPlane, rec + 1);
            cp_async_16(addr + 2u * kWalkPlane, rec + 2);
            stage_side(buf * kWalkThreads + slot, id);
        }
        const unsigned v = __ballot_sync(FULL, valid);
        if (lane == 0) s_cnt[buf][warp] = __popc(v);
    };

    uint32_t next_id = 0;
    {
        const bool v0 = (uint32_t)tid < len;
        stage(0u, v0, v0 ? __ldg(point_list + range.x + tid) : 0u);
        if (kWalkThreads + (uint32_t)tid < len) next_id = __ldg(point_list + range.x + kWalkThreads + tid);
        cp_async_wait_all2();
    }
    __syncthreads();
    const auto consts = make_consts();

    for (uint32_t r = 0; r < nrounds; r++) {
        const uint32_t buf  = r & 1u;
        const uint32_t nidx = (r + 1u) * kWalkThreads + tid;
        if (r + 1u < nrounds) stage(buf ^ 1u, nidx < len, next_id);  // lands while round r is walked
        if (nidx + kWalkThreads < len) next_id = __ldg(point_list + range.x + nidx + kWalkThreads);

        bool da = Ta < 0.0f, db = Tb < 0.0f;
        if (!__all_sync(FULL, da && db)) {
            const uint32_t abase = sbase + buf * kWalkBuf;
            // bounding box of the pixels of the patch that are still accumulating: finished pixels need no more
            // Gaussians, so later rounds cull against a smaller rectangle
            const unsigned lx = (unsigned)(lane & 7), ly = (unsigned)(lane >> 3);
            const unsigned ax = (da && db) ? 255u : lx, bx = (da && db) ? 0u : lx;
            const unsigned ay = !da ? ly : (!db ? ly + 4u : 255u), by = !db ? ly + 4u : (!da ? ly : 0u);
            const float wx0 = (float)(p.patch_x0 + (int)__reduce_min_sync(FULL, ax));
            const float wy0 = (float)(p.patch_y0 + (int)__reduce_min_sync(FULL, ay));
            const float wx1 = (float)(p.patch_x0 + (int)__reduce_max_sync(FULL, bx));
            const float wy1 = (float)(p.patch_y0 + (int)__reduce_max_sync(FULL, by));
#pragma unroll 1
            for (int seg = 0; seg < kWalkWarps; seg++) {
                const uint32_t cnt     = s_cnt[buf][seg];
                const uint32_t segbase = abase + seg * 512u;
                bool           hit_me  = false;
                if ((uint32_t)lane + cnt >= 32u) {
                    const float4 ga = lds128(segbase + lane * 16u);
                    const float4 gb = lds128(segbase + kWalkPlane + lane * 16u);
                    const float  rx = lds32(segbase + 2u * kWalkPlane + lane * 16u + 12u);
                    hit_me = !cull_rect_fast(ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.w, rx, wx0, wy0, wx1, wy1);
                }
                unsigned hits = __ballot_sync(FULL, hit_me);
                while (hits) {
                    const int      top  = top_bit(hits);
                    const uint32_t addr = segbase + top * 16u;
                    hits ^= bit_at(top);
                    const float4 ea = lds128(addr);
                    const float4 eb = lds128(addr + kWalkPlane);
                    const float4 ec = lds128(addr + 2u * kWalkPlane);
                    hit(consts, ea, eb, ec, buf * kWalkThreads + (uint32_t)seg * 32u + (uint32_t)top);
                }
                da = Ta < 0.0f;
                db = Tb < 0.0f;
                if (__all_sync(FULL, da && db)) break;
            }
        }
        cp_async_wait_all2();  // this thread's copies have landed; the barrier publishes everybody's
        if (__syncthreads_and(Ta < 0.0f && Tb < 0.0f)) break;
    }
}

}  // namespace lcgs_b200
