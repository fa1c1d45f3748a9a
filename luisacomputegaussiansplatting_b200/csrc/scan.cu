// scan.cu -- stage 2: inclusive prefix sum of tiles_touched (uint32), single pass with decoupled
// look-back.  Replaces lcpp DeviceScan<>::InclusiveSum (call site
// lcgs/src/gs_tile_splatter/impl.cpp:103-107) and the 4-byte D2H read-back of the last element:
// the grand total (num_rendered) is left in device memory for the following stages.
//
// HBM-bound: 8 bytes per item (one 4-byte read, one 4-byte write), 16-byte vector accesses.
#include "common.cuh"
#include "lookback.cuh"

namespace lcgs_b200 {

__global__ void __launch_bounds__(kScanThreads)
    scan_inclusive_kernel(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, uint32_t n, uint32_t num_tiles,
                          unsigned long long* status, uint32_t* ticket, uint32_t* d_total, int vec_ok)
{
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_warp_sum[kScanThreads / 32];
    __shared__ uint32_t s_tile_prefix;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);  // tiles start in ticket order: look-back cannot deadlock
    __syncthreads();
    const uint32_t tile = s_tile;
    if (tile >= num_tiles) return;
    const uint32_t base = tile * kScanTile + warp * (kScanItems * 32);

    // warp-striped: chunk j of a warp is 128 consecutive items, 4 per lane
    uint32_t v[kScanItems / 4][4];
#pragma unroll
    for (int j = 0; j < kScanItems / 4; j++) {
        const uint32_t e = base + j * 128 + lane * 4;
        if (vec_ok && e + 3 < n) {
            const uint4 q = __ldg(reinterpret_cast<const uint4*>(in + e));
            v[j][0] = q.x; v[j][1] = q.y; v[j][2] = q.z; v[j][3] = q.w;
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++) v[j][k] = (e + k < n) ? __ldg(in + e + k) : 0u;
        }
    }
    // per-thread serial scan inside each chunk, warp scan across lanes, carry across chunks
    uint32_t carry = 0;
    uint32_t excl[kScanItems / 4];
#pragma unroll
    for (int j = 0; j < kScanItems / 4; j++) {
        v[j][1] += v[j][0];
        v[j][2] += v[j][1];
        v[j][3] += v[j][2];
        uint32_t x = v[j][3];
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
            if (lane >= d) x += y;
        }
        excl[j] = carry + x - v[j][3];
        carry += __shfl_sync(0xFFFFFFFFu, x, 31);
    }
    if (lane == 0) s_warp_sum[warp] = carry;
    __syncthreads();

    uint32_t warp_prefix = 0, tile_sum = 0;
#pragma unroll
    for (int w = 0; w < kScanThreads / 32; w++) {
        const uint32_t x = s_warp_sum[w];
        if (w < warp) warp_prefix += x;
        tile_sum += x;
    }

    if (warp == 0) {
        const uint32_t prefix = lookback_warp_u32(status, tile, tile_sum);
        if (lane == 0) {
            s_tile_prefix = prefix;
            if (tile == num_tiles - 1 && d_total) *d_total = prefix + tile_sum;
        }
    }
    __syncthreads();
    const uint32_t add = s_tile_prefix + warp_prefix;

#pragma unroll
    for (int j = 0; j < kScanItems / 4; j++) {
        const uint32_t e = base + j * 128 + lane * 4;
        const uint32_t o = add + excl[j];
        if (vec_ok && e + 3 < n) {
            *reinterpret_cast<uint4*>(out + e) = make_uint4(o + v[j][0], o + v[j][1], o + v[j][2], o + v[j][3]);
        } else {
#pragma unroll
            for (int k = 0; k < 4; k++)
                if (e + k < n) out[e + k] = o + v[j][k];
        }
    }
}

// ---- fused-path variants ----------------------------------------------------------------------
// The fused frame sorts the GAUSSIANS by depth first (3.7 M 8-byte pairs at C3) and emits the
// instances in that order, so that the 17.8 M 12-byte instance pairs only need a stable sort by
// their 13 tile bits (2 radix passes instead of 5).  A stable sort by tile of a list ordered by
// (depth, index) is exactly the order of a stable 64-bit sort of (tile<<32 | depth) keys emitted in
// index order, so sorted keys, sorted values and ranges are bit-identical to the reference's.
//
// scan_compact_kernel: point_offsets (inclusive sum of tiles_touched, the reference's output) AND a
// stable compaction of the Gaussians that touch a tile into (depth bits, index) pairs.  The offsets of
// the emission in depth order are chained inside the emission kernel itself (binning.cu).

struct ScanPair {
    uint32_t a, b;
};

// block-wide exclusive scan of two values per thread (warp shuffles + one shared-memory hop);
// returns the exclusive prefix and the block totals
__device__ __forceinline__ ScanPair block_scan_pair(ScanPair v, ScanPair* s_warp /* [8] */, ScanPair* total)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t  xa = v.a, xb = v.b;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t ya = __shfl_up_sync(0xFFFFFFFFu, xa, d), yb = __shfl_up_sync(0xFFFFFFFFu, xb, d);
        if (lane >= d) { xa += ya; xb += yb; }
    }
    if (lane == 31) s_warp[warp] = ScanPair{ xa, xb };
    __syncthreads();
    ScanPair pre{ 0, 0 }, tot{ 0, 0 };
#pragma unroll
    for (int w = 0; w < kScanThreads / 32; w++) {
        const ScanPair x = s_warp[w];
        if (w < warp) { pre.a += x.a; pre.b += x.b; }
        tot.a += x.a; tot.b += x.b;
    }
    __syncthreads();
    *total = tot;
    return ScanPair{ pre.a + xa - v.a, pre.b + xb - v.b };
}

__global__ void __launch_bounds__(kScanThreads)
    scan_compact_kernel(const uint32_t* __restrict__ tiles_touched, const float* __restrict__ depth, uint32_t n,
                        uint32_t num_tiles, uint32_t* __restrict__ offsets, uint32_t* __restrict__ ckeys,
                        uint32_t* __restrict__ cvals, unsigned long long* status_sum, unsigned long long* status_cnt,
                        uint32_t* ticket, uint32_t* d_total, uint32_t* d_count, const __grid_constant__ SortDigits digits, int vec_ok)
{
    // digit histograms of the depth keys this CTA compacts (the depth sort then skips its histogram kernel)
    __shared__ uint32_t s_hist[kCompactHistPasses * kMaxRadix];
    // the CTA's compacted (key, index) pairs, staged so that they leave as two coalesced runs
    __shared__ uint32_t s_key[kCompactTile], s_idx[kCompactTile];
    const bool          do_hist = digits.hist != nullptr;
    const int           nbins   = do_hist ? (digits.num_passes << digits.radix_bits) : 0;
    for (int k = threadIdx.x; k < nbins; k += kScanThreads) s_hist[k] = 0u;
    __shared__ uint32_t s_tile;
    __shared__ ScanPair s_warp[kScanThreads / 32];
    __shared__ uint32_t s_prefix[2];
    const int tid = threadIdx.x;
    // Persistent CTAs: tiles are taken by ticket (so they start in order and the look-back cannot deadlock), and a
    // CTA's digit histograms are flushed once at the end instead of once per tile -- with one CTA per tile the
    // flushes were ~1500 global atomics x 2800 tiles on 2048 addresses.
    for (;;) {
    __syncthreads();  // s_tile, s_prefix, s_key / s_idx of the previous tile are no longer read
    if (tid == 0) s_tile = atomicAdd(ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    if (tile >= num_tiles) break;
    // blocked arrangement: thread t owns items [base + t*8, +8) -> two 16-byte loads per array; the depths
    // are requested up front for every item (4 B each), not one dependent load per touching Gaussian
    const uint32_t e0 = tile * kCompactTile + tid * kCompactItems;
    uint32_t       v[kCompactItems], dk[kCompactItems];
    if (vec_ok && e0 + kCompactItems <= n) {
        const uint4 q0 = __ldg(reinterpret_cast<const uint4*>(tiles_touched + e0));
        const uint4 q1 = __ldg(reinterpret_cast<const uint4*>(tiles_touched + e0) + 1);
        const uint4 d0 = __ldg(reinterpret_cast<const uint4*>(depth + e0));
        const uint4 d1 = __ldg(reinterpret_cast<const uint4*>(depth + e0) + 1);
        v[0] = q0.x; v[1] = q0.y; v[2] = q0.z; v[3] = q0.w; v[4] = q1.x; v[5] = q1.y; v[6] = q1.z; v[7] = q1.w;
        dk[0] = d0.x; dk[1] = d0.y; dk[2] = d0.z; dk[3] = d0.w; dk[4] = d1.x; dk[5] = d1.y; dk[6] = d1.z; dk[7] = d1.w;
    } else {
#pragma unroll
        for (int k = 0; k < kCompactItems; k++) {
            v[k]  = (e0 + k < n) ? __ldg(tiles_touched + e0 + k) : 0u;
            dk[k] = (e0 + k < n) ? __float_as_uint(__ldg(depth + e0 + k)) : 0u;
        }
    }
    ScanPair mine{ 0, 0 };
#pragma unroll
    for (int k = 0; k < kCompactItems; k++) {
        mine.a += v[k];
        mine.b += v[k] > 0u ? 1u : 0u;
    }
    ScanPair       tot;
    const ScanPair excl = block_scan_pair(mine, s_warp, &tot);
    // two chains (instance sum, touching-Gaussian count), one warp each; the other warps stage meanwhile
    if (tid < 64) {
        const uint32_t pre = (tid < 32) ? lookback_warp_u32(status_sum, tile, tot.a) : lookback_warp_u32(status_cnt, tile, tot.b);
        if ((tid & 31) == 0) s_prefix[tid >> 5] = pre;
    }
    // stable compaction inside the CTA: slots are handed out in index order
    uint32_t sum = excl.a, slot = excl.b;
    uint32_t out[kCompactItems];
#pragma unroll
    for (int k = 0; k < kCompactItems; k++) {
        sum += v[k];
        out[k] = sum;
        if (v[k] > 0u) {
            s_key[slot] = dk[k] - kDepthKeyBase;
            s_idx[slot] = e0 + k;
            slot++;
        }
    }
    __syncthreads();
    const uint32_t base_sum = s_prefix[0], base_cnt = s_prefix[1];
    if (tile == num_tiles - 1 && tid == 0) {
        *d_total = base_sum + tot.a;
        *d_count = base_cnt + tot.b;
    }
    if (vec_ok && e0 + kCompactItems <= n) {
        reinterpret_cast<uint4*>(offsets + e0)[0] = make_uint4(base_sum + out[0], base_sum + out[1], base_sum + out[2], base_sum + out[3]);
        reinterpret_cast<uint4*>(offsets + e0)[1] = make_uint4(base_sum + out[4], base_sum + out[5], base_sum + out[6], base_sum + out[7]);
    } else {
#pragma unroll
        for (int k = 0; k < kCompactItems; k++)
            if (e0 + k < n) offsets[e0 + k] = base_sum + out[k];
    }
    for (uint32_t i = tid; i < tot.b; i += kScanThreads) {
        const uint32_t key = s_key[i];
        ckeys[base_cnt + i] = key;
        cvals[base_cnt + i] = s_idx[i];
        if (do_hist) {
#pragma unroll
            for (int p = 0; p < kCompactHistPasses; p++)
                if (p < digits.num_passes) atomicAdd(&s_hist[(p << digits.radix_bits) + ((key >> digits.shift[p]) & digits.mask[p])], 1u);
        }
    }
    }  // tile loop
    if (do_hist) {
        __syncthreads();
        for (int k = threadIdx.x; k < nbins; k += kScanThreads) {
            const uint32_t c = s_hist[k];
            if (c) atomicAdd(digits.hist + k, c);
        }
    }
}

int launch_scan_compact(lcgs_b200_ctx* ctx, const uint32_t* tiles_touched, const float* depth, int P, uint32_t* offsets,
                        uint32_t* ckeys, uint32_t* cvals, uint32_t* d_total, uint32_t* d_count, const FramePlan& fp,
                        cudaStream_t s)
{
    if (P <= 0) {
        LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(d_total, 0, sizeof(uint32_t), s));
        LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(d_count, 0, sizeof(uint32_t), s));
        return LCGS_B200_OK;
    }
    // 16-byte aligned buffers (any cudaMalloc'ed array) take the vector path, sub-allocated ones the scalar one
    const int vec_ok = ((((uintptr_t)tiles_touched) | ((uintptr_t)offsets) | ((uintptr_t)depth)) & 15) == 0;
    const uint32_t tiles = (uint32_t)compact_tiles(P);
    const uint32_t max_blocks = (uint32_t)ctx->num_sms * (uint32_t)LCGS_TUNE_INT("LCGS_SCAN_CTAS", 6);  // persistent: 6 x 256 threads per SM
    scan_compact_kernel<<<tiles < max_blocks ? tiles : max_blocks, kScanThreads, 0, s>>>(tiles_touched, depth, (uint32_t)P, tiles, offsets, ckeys, cvals,
                                                       fp.scan_sum, fp.scan_count, fp.scan_ticket, d_total, d_count,
                                                       producer_digits(fp.depth), vec_ok);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_scan(lcgs_b200_ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, uint32_t* d_total, cudaStream_t s)
{
    if (n == 0) {
        if (d_total) LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(d_total, 0, sizeof(uint32_t), s));
        return LCGS_B200_OK;
    }
    LCGS_REQUIRE(ctx, n < 0xFFFFFFFFull, "scan: more than 2^32-1 items");
    const uint32_t tiles = (uint32_t)((n + kScanTile - 1) / kScanTile);
    int            rc    = ws_reserve(ctx, ctx->scan_ws, (size_t)tiles * sizeof(unsigned long long));
    if (rc) return rc;
    LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(ctx->scan_ws.ptr, 0, (size_t)tiles * sizeof(unsigned long long), s));
    uint32_t* ticket = ctx->d_scalars + LCGS_SCALAR_SCAN_TICKET;
    LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(ticket, 0, sizeof(uint32_t), s));
    const int vec_ok = (((uintptr_t)in | (uintptr_t)out) & 15) == 0;
    scan_inclusive_kernel<<<tiles, kScanThreads, 0, s>>>(in, out, (uint32_t)n, tiles,
                                                         (unsigned long long*)ctx->scan_ws.ptr, ticket, d_total, vec_ok);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
