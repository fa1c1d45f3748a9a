// binning.cu -- stage 3 (key duplication) and stage 5a (tile ranges), plus the buffer filler.
//
//  * duplicate_keys_kernel replaces shad_copy_with_keys (lcgs/src/gs_tile_splatter/shader.cpp:26-69)
//    and the two zero-fills in front of it (impl.cpp:117-118, pure overhead: every slot below
//    num_rendered is overwritten).  The reference lets ONE thread write all tiles of a Gaussian
//    serially; near-plane Gaussians cover thousands of tiles, so here a warp expands its 32
//    Gaussians cooperatively: lanes walk the warp's contiguous output range, find the owning
//    Gaussian by a shuffle binary search over the warp-local prefix, and store fully coalesced.
//  * tile_ranges_kernel replaces shad_get_ranges (shader.cpp:71-100).
//
// Both are HBM-bound integer work: 12 bytes written per instance, 8 bytes read per instance.
#include "common.cuh"
#include "lookback.cuh"

namespace lcgs_b200 {

__global__ void __launch_bounds__(256)
    duplicate_keys_kernel(int P, uint32_t gx, uint32_t gy, uint32_t row0, uint32_t row1,
                          const float2* __restrict__ means_pix, const uint32_t* __restrict__ offsets,
                          const int32_t* __restrict__ radii, const float* __restrict__ depth,
                          unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals, size_t capacity)
{
    const int      lane        = threadIdx.x & 31;
    const long     warp_global = ((long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long     num_warps   = ((long)gridDim.x * blockDim.x) >> 5;
    const unsigned FULL        = 0xFFFFFFFFu;

    for (long base = warp_global * 32; base < P; base += num_warps * 32) {
        const long i   = base + lane;
        uint32_t   cnt = 0, x0 = 0, y0 = 0, w = 1, dbits = 0, incl = 0;
        if (i < P) {
            incl             = __ldg(offsets + i);
            const int radius = __ldg(radii + i);
            if (radius > 0) {
                const float2   m = __ldg(means_pix + i);
                const TileRect r = get_rect(m.x, m.y, radius, gx, gy, row0, row1);
                x0               = r.x0;
                y0               = r.y0;
                w                = r.x1 - r.x0;
                cnt              = w * (r.y1 - r.y0);
                dbits            = float_bits(__ldg(depth + i));
                if (w == 0) w = 1;
            }
        }
        // exclusive global offset of Gaussian i = offsets[i-1] (0 for i == 0), shader.cpp:42-46
        uint32_t excl = __shfl_up_sync(FULL, incl, 1);
        if (lane == 0) excl = (base > 0) ? __ldg(offsets + base - 1) : 0u;
        // warp-local exclusive prefix of the per-Gaussian counts
        uint32_t x = cnt;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(FULL, x, d);
            if (lane >= d) x += y;
        }
        const uint32_t loc   = x - cnt;
        const uint32_t total = __shfl_sync(FULL, x, 31);

        for (uint32_t p0 = 0; p0 < total; p0 += 32) {
            const uint32_t p = p0 + lane;
            // owner = largest lane l with loc_l <= p (zero-count lanes share their successor's loc and
            // are skipped because the search prefers the higher lane)
            int l = 0;
#pragma unroll
            for (int step = 16; step >= 1; step >>= 1) {
                const uint32_t v = __shfl_sync(FULL, loc, l + step);
                if (v <= p) l += step;
            }
            const uint32_t o_loc   = __shfl_sync(FULL, loc, l);
            const uint32_t o_excl  = __shfl_sync(FULL, excl, l);
            const uint32_t o_x0    = __shfl_sync(FULL, x0, l);
            const uint32_t o_y0    = __shfl_sync(FULL, y0, l);
            const uint32_t o_w     = __shfl_sync(FULL, w, l);
            const uint32_t o_dbits = __shfl_sync(FULL, dbits, l);
            if (p < total) {
                const uint32_t k  = p - o_loc;  // index inside the owner's rect, row-major
                const uint32_t ry = k / o_w;
                const uint32_t rx = k - ry * o_w;
                const uint32_t tile = (o_x0 + rx) + (o_y0 + ry - row0) * gx;
                const size_t   dst  = (size_t)o_excl + k;
                if (dst < capacity) {
                    keys[dst] = ((unsigned long long)tile << 32) | (unsigned long long)o_dbits;
                    vals[dst] = (uint32_t)(base + l);
                }
            }
        }
    }
}

// Fused-path emission: Gaussians are visited in depth order (sorted (depth key, index) pairs); rects are
// the packed tile rects preprocess wrote (x0 | y0<<16, w | h<<16).  One kernel does what used to be two
// (an inclusive scan of the tile counts in depth order, then the emission): CTAs take tiles of 1024
// Gaussians by ticket, chain the tile's instance count to its predecessors with a decoupled look-back
// (lookback.cuh) and expand their Gaussians warp-cooperatively as above, 32 Gaussians per warp and step.
// A ticket is only taken when the CTA is ready to load, count and publish at once: a tile that is held
// back (e.g. taken ahead of time to prefetch it) stalls the look-back of every tile behind it.
constexpr int kEmitWarps = kEmitThreads / 32;  // kEmitThreads, kEmitTile: frame_plan.cuh

__device__ __forceinline__ void red_shared_add(uint32_t addr, uint32_t v)
{
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// Gaussians that cover more than `big_threshold` tiles are not expanded by the warp that owns them (one warp walking a
// 10 000-tile rect is the whole kernel's tail: on a sparse band of the 8K frame 1 % of the Gaussians hold a third of the
// instances, and a single warp was found emitting 52 000 instances while the rest of the GPU idled).  The warp only
// reserves their output range (offsets are chained over the TRUE counts) and appends (entry, piece) work items;
// emit_big_kernel then expands all pieces of kBigPiece instances, one CTA per piece, perfectly balanced (BigLists,
// frame_plan.cuh).

// Tile-bit digit histograms of up to 32 emitted keys (one per lane; every lane of the warp must call).  Consecutive lanes
// emit consecutive tiles of one Gaussian, so the upper digit is counted once per run of equal digits.
struct EmitHist {
    uint32_t hist_addr, hist1_addr, m0, m1;
    int      sh0, sh1;
    bool     on, two_digits;
};
__device__ __forceinline__ void emit_hist_update(const EmitHist& h, bool emit, uint32_t tile, int lane, unsigned le_mask)
{
    const unsigned FULL = 0xFFFFFFFFu;
    if (!h.on) return;
    if (emit) red_shared_add(h.hist_addr + (((tile >> h.sh0) & h.m0) << 2), 1u);
    if (h.two_digits) {
        const uint32_t d1      = (tile >> h.sh1) & h.m1;
        const uint32_t prev    = __shfl_up_sync(FULL, d1, 1);
        const bool     was     = __shfl_up_sync(FULL, emit ? 1 : 0, 1) != 0;
        const bool     lead    = emit && (lane == 0 || prev != d1 || !was);
        const unsigned leaders = __ballot_sync(FULL, lead);
        const unsigned emits   = __ballot_sync(FULL, emit);
        if (lead) {
            // the run ends at the next leader or at the first lane above that does not emit
            const unsigned stop = (leaders | ~emits) & ~le_mask;
            const int      end  = stop ? __ffs(stop) - 1 : 32;
            red_shared_add(h.hist1_addr + (d1 << 2), (uint32_t)(end - lane));
        }
    }
}

// BIG: with the side path for big Gaussians (frames / bands of at least kBigPathMinTiles tiles, where one Gaussian can
// cover thousands of them); without it the kernel is the plain warp-cooperative expansion, which is 12 % faster on the
// 1080p frame, whose largest Gaussian covers about a thousand tiles.
constexpr uint32_t kBigPathMinTiles = 12288;

// HIST2: "both digit histograms of the tile sort are accumulated" is a compile-time fact (the fused frame of any picture
// up to 16 384 tiles): the uniform tests of it leave the expansion loop.
template <bool BIG, bool EXACT_DIV, bool HIST2 = false>
__device__ __forceinline__ void duplicate_keys_sorted_body(const uint32_t* __restrict__ d_m, uint32_t m_capacity, uint32_t gx, uint32_t row0,
                                                           const SortedPairsU32& sorted, const uint2* __restrict__ rects,
                                                           unsigned long long* status, uint32_t* ticket,
                                                           unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals,
                                                           size_t capacity, const SortDigits& digits, const BigLists& big)
{
    constexpr bool exact_div = EXACT_DIV;  // index inside a rect -> (x, y) by multiply-high instead of a division
    // digit histograms of the tile bits of the emitted keys (two passes at most: the tile sort then skips
    // its histogram kernel).  Consecutive lanes emit consecutive tiles of one Gaussian, so the upper digit
    // is aggregated per run of equal digits.
    __shared__ uint32_t s_hist[kEmitHistPasses * kMaxRadix];
    __shared__ uint32_t s_wsum[kEmitWarps];
    __shared__ uint32_t s_base;
    __shared__ uint32_t s_tk;
    const bool     do_hist = HIST2 || digits.hist != nullptr;
    const int      nbins   = do_hist ? (digits.num_passes << digits.radix_bits) : 0;
    const int      tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned FULL = 0xFFFFFFFFu;
    for (int k = tid; k < nbins; k += kEmitThreads) s_hist[k] = 0u;
    const uint32_t hist_addr = (uint32_t)__cvta_generic_to_shared(s_hist);
    const int      sh0 = digits.shift[0] - 32, sh1 = digits.shift[1] - 32;
    const uint32_t m0 = digits.mask[0], m1 = digits.mask[1], hist1_addr = hist_addr + (4u << digits.radix_bits);
    const bool     two_digits = HIST2 || digits.num_passes > 1;

    uint32_t M = *d_m;
    if (M > m_capacity) M = m_capacity;
    const uint32_t num_tiles           = (M + kEmitTile - 1) / kEmitTile;
    const bool     in_alt              = sorted_in_alt(sorted, M);
    const uint32_t* __restrict__ order = in_alt ? sorted.alt_vals : sorted.vals;
    const uint32_t* __restrict__ skeys = in_alt ? sorted.alt_keys : sorted.keys;
    const unsigned le_mask             = (2u << lane) - 1u;  // lanes 0..lane (all ones for lane 31)

    for (;;) {
        __syncthreads();  // s_tk, s_wsum and s_base of the previous tile are no longer read
        if (tid == 0) s_tk = atomicAdd(ticket, 1u);
        __syncthreads();
        const uint32_t t = s_tk;
        if (t >= num_tiles) break;

        // ---- load: (index, depth key) coalesced, then the rect gathers, all chunks in flight together ----
        const uint32_t k0 = t * kEmitTile + warp * (32 * kEmitItems) + lane;
        uint32_t       idx[kEmitItems], dbits[kEmitItems], xy0[kEmitItems], w[kEmitItems], cnt[kEmitItems];
#pragma unroll
        for (int c = 0; c < kEmitItems; c++) {
            const uint32_t k = k0 + 32 * c;
            idx[c]           = 0xFFFFFFFFu;  // none
            dbits[c]         = 0u;
            if (k < M) {
                idx[c]   = __ldg(order + k);
                dbits[c] = __ldg(skeys + k) + kDepthKeyBase;  // keys are sorted relative to the base
            }
        }
#pragma unroll
        for (int c = 0; c < kEmitItems; c++) {
            uint2 r = make_uint2(0u, 0u);
            if (idx[c] != 0xFFFFFFFFu) r = __ldg(rects + idx[c]);
            xy0[c] = r.x;
            w[c]   = r.y & 0xFFFFu;
            cnt[c] = w[c] * (r.y >> 16);
            if (w[c] == 0u) w[c] = 1u;
        }
        // ---- count: inclusive scan inside each chunk, chunk bases inside the warp, totals across the CTA ----
        uint32_t incl[kEmitItems], cbase[kEmitItems], wtot = 0;
#pragma unroll
        for (int c = 0; c < kEmitItems; c++) {
            uint32_t x = cnt[c];
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(FULL, x, d);
                if (lane >= d) x += y;
            }
            incl[c]  = x;
            cbase[c] = wtot;
            wtot += __shfl_sync(FULL, x, 31);
        }
        if (lane == 0) s_wsum[warp] = wtot;
        __syncthreads();
        uint32_t wpre = 0, ttot = 0;
#pragma unroll
        for (int v = 0; v < kEmitWarps; v++) {
            const uint32_t c = s_wsum[v];
            if (v < warp) wpre += c;
            ttot += c;
        }
        if (warp == 0) {
            const uint32_t pre = lookback_warp_u32(status, t, ttot);
            if (lane == 0) s_base = pre;
        }
        __syncthreads();
        const uint32_t wbase = s_base + wpre;  // output offset of this warp's first instance

        // ---- emit: a chunk's instances are one contiguous run of the output, minus the ranges of its big Gaussians,
        // which are handed to emit_big_kernel.  Slot p of the chunk's INLINE run belongs to the lane `l` whose inline
        // run contains it and goes to that Gaussian's true output offset + (p - start of its inline run). ----------
#pragma unroll
        for (int c = 0; c < kEmitItems; c++) {
            const bool     valid  = idx[c] != 0xFFFFFFFFu;
            const uint32_t excl0  = wbase + cbase[c];                     // first output slot of the chunk
            const uint32_t texcl  = excl0 + incl[c] - cnt[c];             // first output slot of this lane's Gaussian
            const bool     is_big = BIG && valid && cnt[c] > big.threshold;
            if (is_big) {
                const uint32_t np = (cnt[c] + kBigPiece - 1) / kBigPiece;
                const uint32_t e  = atomicAdd(big.counters, 1u);
                const uint32_t pb = atomicAdd(big.counters + 1, np);
                if (e < big.entry_capacity) {
                    big.entries[e] = BigEntry{ texcl, cnt[c], xy0[c], w[c], dbits[c], idx[c], 0u, 0u };
                    for (uint32_t k = 0; k < np; k++)
                        if (pb + k < big.piece_capacity) big.pieces[pb + k] = make_uint2(e, k);
                }
            }
            const bool     any_big = BIG && __any_sync(FULL, is_big);
            const uint32_t icnt    = is_big ? 0u : cnt[c];
            uint32_t       iincl   = incl[c];
            if (any_big) {  // inline counts need their own scan
                iincl = icnt;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const uint32_t y = __shfl_up_sync(FULL, iincl, d);
                    if (lane >= d) iincl += y;
                }
            }
            const uint32_t total = __shfl_sync(FULL, iincl, 31);
            const uint32_t loc   = iincl - icnt;
            // q = j / w as a multiply-high (exact while j * w < 2^32, checked on the host for the grid)
            const uint32_t magic = (uint32_t)(0x100000000ull / w[c]) + 1u;
            // Every compacted Gaussian touches a tile, so (without big ones) owners are consecutive lanes and an output
            // slot finds its owner by counting the Gaussian starts at or before it: one ballot, one OR-reduction, two popc.
            const bool dense = exact_div && !any_big && __all_sync(FULL, !valid || cnt[c] > 0u);
            for (uint32_t p0 = 0; p0 < total; p0 += 32) {
                const uint32_t p = p0 + lane;
                int            l;
                if (dense) {
                    const unsigned before = __ballot_sync(FULL, valid && loc <= p0);
                    const unsigned starts = __reduce_or_sync(FULL, (valid && loc > p0 && loc - p0 < 32u) ? 1u << (loc - p0) : 0u);
                    l                     = __popc(before) - 1 + __popc(starts & le_mask);
                } else {
                    // owner = largest lane with loc <= p (zero-count lanes share their successor's loc and
                    // are skipped because the search prefers the higher lane)
                    l = 0;
#pragma unroll
                    for (int step = 16; step >= 1; step >>= 1) {
                        const uint32_t v = __shfl_sync(FULL, loc, l + step);
                        if (v <= p) l += step;
                    }
                }
                const uint32_t o_loc   = __shfl_sync(FULL, loc, l);
                const uint32_t o_texcl = BIG ? __shfl_sync(FULL, texcl, l) : 0u;
                const uint32_t o_xy0   = __shfl_sync(FULL, xy0[c], l);
                const uint32_t o_w     = __shfl_sync(FULL, w[c], l);
                const uint32_t o_magic = __shfl_sync(FULL, magic, l);
                const uint32_t o_dbits = __shfl_sync(FULL, dbits[c], l);
                const uint32_t o_idx   = __shfl_sync(FULL, idx[c], l);
                // every lane computes (sync intrinsics below stay convergent with the full mask); lanes past the
                // end of the run or of the list capacity -- a suffix of the warp -- neither store nor count
                const uint32_t j    = p - o_loc;
                const uint32_t ry   = exact_div ? (o_w == 1u ? j : __umulhi(j, o_magic)) : j / o_w;  // magic wraps for w == 1
                const uint32_t rx   = j - ry * o_w;
                const uint32_t tile = ((o_xy0 & 0xFFFFu) + rx) + ((o_xy0 >> 16) + ry - row0) * gx;
                const size_t   dst  = BIG ? (size_t)o_texcl + j : (size_t)excl0 + p;  // without gaps the chunk's run is contiguous
                const bool     emit = p < total && dst < capacity;
                if (emit) {
                    keys[dst] = ((unsigned long long)tile << 32) | (unsigned long long)o_dbits;
                    vals[dst] = o_idx;
                }
                if (do_hist) {
                    if (emit) red_shared_add(hist_addr + (((tile >> sh0) & m0) << 2), 1u);
                    if (two_digits) {
                        // consecutive lanes emit consecutive tiles: runs of equal upper digits are counted by
                        // their first lane (MATCH.ANY is slow); emitting lanes are a prefix of the warp
                        const uint32_t d1      = (tile >> sh1) & m1;
                        const uint32_t prev    = __shfl_up_sync(FULL, d1, 1);
                        const bool     lead    = emit && (lane == 0 || prev != d1);
                        const unsigned leaders = __ballot_sync(FULL, lead);
                        const int      n_emit  = __popc(__ballot_sync(FULL, emit));
                        if (lead) {
                            const unsigned above = leaders & ~le_mask;
                            const int      end   = above ? __ffs(above) - 1 : n_emit;
                            red_shared_add(hist1_addr + (d1 << 2), (uint32_t)(end - lane));
                        }
                    }
                }
            }
        }
    }
    if (do_hist) {
        __syncthreads();
        for (int k = tid; k < nbins; k += kEmitThreads) {
            const uint32_t c = s_hist[k];
            if (c) atomicAdd(digits.hist + k, c);
        }
    }
}

// Two entry points over one body: the plain kernel takes no big-list parameters at all (with them in its parameter
// block the compiler re-loaded kernel constants inside the expansion loop: +30 % instructions per step).
template <bool EXACT_DIV, bool HIST2 = false>
__global__ void __launch_bounds__(kEmitThreads)
    duplicate_keys_sorted_kernel(const uint32_t* __restrict__ d_m, uint32_t m_capacity, uint32_t gx, uint32_t row0,
                                 const __grid_constant__ SortedPairsU32 sorted, const uint2* __restrict__ rects,
                                 unsigned long long* status, uint32_t* ticket, unsigned long long* __restrict__ keys,
                                 uint32_t* __restrict__ vals, size_t capacity, const __grid_constant__ SortDigits digits)
{
    duplicate_keys_sorted_body<false, EXACT_DIV, HIST2>(d_m, m_capacity, gx, row0, sorted, rects, status, ticket, keys, vals, capacity, digits,
                                                 BigLists{});
}

template <bool EXACT_DIV>
__global__ void __launch_bounds__(kEmitThreads, 5)
    duplicate_keys_sorted_big_kernel(const uint32_t* __restrict__ d_m, uint32_t m_capacity, uint32_t gx, uint32_t row0,
                                     const __grid_constant__ SortedPairsU32 sorted, const uint2* __restrict__ rects,
                                     unsigned long long* status, uint32_t* ticket, unsigned long long* __restrict__ keys,
                                     uint32_t* __restrict__ vals, size_t capacity, const __grid_constant__ SortDigits digits,
                                     const __grid_constant__ BigLists big)
{
    duplicate_keys_sorted_body<true, EXACT_DIV>(d_m, m_capacity, gx, row0, sorted, rects, status, ticket, keys, vals, capacity, digits, big);
}

// One CTA per (entry, piece): kBigPiece consecutive instances of one big Gaussian, coalesced.
__global__ void __launch_bounds__(kEmitThreads)
    emit_big_kernel(uint32_t gx, uint32_t row0, unsigned long long* __restrict__ keys, uint32_t* __restrict__ vals, size_t capacity,
                    const __grid_constant__ SortDigits digits, bool exact_div, const __grid_constant__ BigLists big)
{
    __shared__ uint32_t s_hist[kEmitHistPasses * kMaxRadix];
    const bool     do_hist = digits.hist != nullptr;
    const int      nbins   = do_hist ? (digits.num_passes << digits.radix_bits) : 0;
    const int      tid = threadIdx.x, lane = tid & 31;
    const unsigned le_mask = (2u << lane) - 1u;
    for (int k = tid; k < nbins; k += kEmitThreads) s_hist[k] = 0u;
    const uint32_t hist_addr = (uint32_t)__cvta_generic_to_shared(s_hist);
    const EmitHist eh{ hist_addr, hist_addr + (4u << digits.radix_bits), digits.mask[0], digits.mask[1],
                       digits.shift[0] - 32, digits.shift[1] - 32, do_hist, digits.num_passes > 1 };
    __syncthreads();
    uint32_t np = big.counters[1];
    if (np > big.piece_capacity) np = big.piece_capacity;
    for (uint32_t q = blockIdx.x; q < np; q += gridDim.x) {
        const uint2 pc = __ldg(big.pieces + q);
        if (pc.x >= big.entry_capacity) continue;
        const BigEntry e     = big.entries[pc.x];
        const uint32_t magic = (uint32_t)(0x100000000ull / e.w) + 1u;
        const uint32_t j0 = pc.y * kBigPiece, j1 = min(e.cnt, j0 + kBigPiece);
        for (uint32_t jb = j0; jb < j1; jb += kEmitThreads) {  // uniform trip count: the histogram helper is warp-synchronous
            const uint32_t j    = jb + tid;
            const uint32_t ry   = exact_div ? (e.w == 1u ? j : __umulhi(j, magic)) : j / e.w;
            const uint32_t rx   = j - ry * e.w;
            const uint32_t tile = ((e.xy0 & 0xFFFFu) + rx) + ((e.xy0 >> 16) + ry - row0) * gx;
            const size_t   dst  = (size_t)e.dst + j;
            const bool     emit = j < j1 && dst < capacity;
            if (emit) {
                keys[dst] = ((unsigned long long)tile << 32) | (unsigned long long)e.dbits;
                vals[dst] = e.idx;
            }
            emit_hist_update(eh, emit, tile, lane, le_mask);
        }
    }
    if (do_hist) {
        __syncthreads();
        for (int k = tid; k < nbins; k += kEmitThreads) {
            const uint32_t c = s_hist[k];
            if (c) atomicAdd(digits.hist + k, c);
        }
    }
}

__global__ void __launch_bounds__(256)
    tile_ranges_kernel(const unsigned long long* __restrict__ keys, size_t n_host, const uint32_t* __restrict__ d_n,
                       size_t capacity, uint32_t* __restrict__ ranges, uint32_t num_tiles)
{
    size_t n = n_host;
    if (d_n) {
        n = *d_n;
        if (n > capacity) n = capacity;
    }
    // boundary between sorted positions k-1 and k (shad_get_ranges, shader.cpp:73-99)
    auto boundary = [&](size_t k, uint32_t prev, uint32_t cur) {
        if (k == 0) {
            if (cur < num_tiles) ranges[2 * cur] = 0u;
        } else if (cur != prev) {
            if (prev < num_tiles) ranges[2 * prev + 1] = (uint32_t)k;
            if (cur < num_tiles) ranges[2 * cur] = (uint32_t)k;
        }
        if (k == n - 1 && cur < num_tiles) ranges[2 * cur + 1] = (uint32_t)n;
    };
    // four keys per thread and iteration: two 16-byte loads plus the predecessor's tile id
    const size_t stride = (size_t)gridDim.x * blockDim.x * 4;
    for (size_t k = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4; k < n; k += stride) {
        if (k + 3 < n) {
            const ulonglong2 a = __ldg(reinterpret_cast<const ulonglong2*>(keys + k));
            const ulonglong2 b = __ldg(reinterpret_cast<const ulonglong2*>(keys + k) + 1);
            const uint32_t   t0 = (uint32_t)(a.x >> 32), t1 = (uint32_t)(a.y >> 32), t2 = (uint32_t)(b.x >> 32), t3 = (uint32_t)(b.y >> 32);
            const uint32_t   tp = k ? (uint32_t)(__ldg(keys + k - 1) >> 32) : 0u;
            boundary(k, tp, t0);
            boundary(k + 1, t0, t1);
            boundary(k + 2, t1, t2);
            boundary(k + 3, t2, t3);
        } else {
            uint32_t prev = k ? (uint32_t)(__ldg(keys + k - 1) >> 32) : 0u;
            for (size_t j = k; j < n; j++) {
                const uint32_t cur = (uint32_t)(__ldg(keys + j) >> 32);
                boundary(j, prev, cur);
                prev = cur;
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(256) fill_kernel(T* __restrict__ buf, size_t n, T v)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) buf[k] = v;
}

int launch_duplicate_keys(lcgs_b200_ctx* ctx, int P, int W, int H, const float* means_2d, const uint32_t* offsets,
                          const int32_t* radii, const float* depth, uint64_t* keys, uint32_t* vals, size_t capacity,
                          int row0, int row1, cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    const uint32_t gx = (uint32_t)((W + 15) / 16), gy = (uint32_t)((H + 15) / 16);
    const long     warps_needed = ((long)P + 31) / 32;
    long           blocks       = (warps_needed + 7) / 8;
    const long     max_blocks   = (long)ctx->num_sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    duplicate_keys_kernel<<<(unsigned)blocks, 256, 0, s>>>(P, gx, gy, (uint32_t)row0, row1 < 0 ? gy : (uint32_t)row1,
                                                          reinterpret_cast<const float2*>(means_2d), offsets, radii,
                                                          depth, reinterpret_cast<unsigned long long*>(keys), vals,
                                                          capacity);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_duplicate_keys_sorted(lcgs_b200_ctx* ctx, const uint32_t* d_m, int P, int W, int H, int num_rows,
                                 const SortedPairsU32& sorted, const uint2* rects, uint64_t* keys, uint32_t* vals,
                                 size_t capacity, int row0, const FramePlan& fp, cudaStream_t s)
{
    if (P <= 0) return LCGS_B200_OK;
    SortDigits dg = producer_digits(fp.tile);
    if (dg.num_passes < 2) dg.shift[1] = 32;  // unused, but keep the kernel's shift amounts in range
    const uint32_t gx = (uint32_t)((W + 15) / 16);
    // index inside a rect / rect width as a multiply-high: exact while j * w < 2^32; j < w * h with w <= gx and
    // h <= gy, so it is enough that gx * gx * gy stays below 2^32 (an 8K frame: 480 * 480 * 270 = 6.2e7).
    // Rect heights are bounded by the band's row count, so a band of a huge frame keeps the fast path; the general
    // path (division, owner search by shuffle) is covered by the extreme-aspect test (640000 x 48 pixels).
    const uint32_t gy        = (uint32_t)(num_rows > 0 ? num_rows : (H + 15) / 16);
    const bool     exact_div = (unsigned long long)gx * gx * gy < 0x100000000ull;
    const uint32_t tiles     = (uint32_t)emit_tiles(P);
    // persistent CTAs; tiles are handed out by ticket, so CTAs that are not resident yet hold nothing back
    const uint32_t max_blocks = (uint32_t)ctx->num_sms * (uint32_t)LCGS_TUNE_INT("LCGS_EMIT_CTAS", 6);
    const uint32_t blocks     = tiles < max_blocks ? tiles : max_blocks;
    const bool big_path = (unsigned long long)gx * gy >= (unsigned long long)LCGS_TUNE_INT("LCGS_EMIT_BIG_MIN_TILES", (int)kBigPathMinTiles);
    auto* const k64 = reinterpret_cast<unsigned long long*>(keys);
    if (big_path) {
        auto kern = exact_div ? duplicate_keys_sorted_big_kernel<true> : duplicate_keys_sorted_big_kernel<false>;
        kern<<<blocks, kEmitThreads, 0, s>>>(d_m, (uint32_t)P, gx, (uint32_t)row0, sorted, rects, fp.emit_status, fp.emit_ticket, k64, vals,
                                             capacity, dg, fp.big);
    } else {
        auto kern = exact_div ? duplicate_keys_sorted_kernel<true> : duplicate_keys_sorted_kernel<false>;
        if (exact_div && dg.hist && dg.num_passes == 2 && LCGS_TUNE_INT("LCGS_EMIT_HIST2", 1)) kern = duplicate_keys_sorted_kernel<true, true>;
        kern<<<blocks, kEmitThreads, 0, s>>>(d_m, (uint32_t)P, gx, (uint32_t)row0, sorted, rects, fp.emit_status, fp.emit_ticket, k64, vals,
                                             capacity, dg);
    }
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    if (big_path) {
        emit_big_kernel<<<max_blocks, kEmitThreads, 0, s>>>(gx, (uint32_t)row0, k64, vals, capacity, dg, exact_div, fp.big);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    }
    return LCGS_B200_OK;
}

int launch_ranges(lcgs_b200_ctx* ctx, const uint64_t* keys, size_t n_host, const uint32_t* d_n, size_t capacity,
                  uint32_t* ranges, int num_tiles, cudaStream_t s, bool cleared)
{
    if (num_tiles <= 0) return LCGS_B200_OK;
    if (!cleared) LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(ranges, 0, (size_t)num_tiles * 2 * sizeof(uint32_t), s));
    const size_t bound = d_n ? capacity : n_host;
    if (bound == 0) return LCGS_B200_OK;
    LCGS_REQUIRE(ctx, (((uintptr_t)keys) & 15) == 0, "tile_ranges: keys must be 16-byte aligned");
    size_t       blocks     = (bound + 4095) / 4096;
    const size_t max_blocks = (size_t)ctx->num_sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    tile_ranges_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const unsigned long long*>(keys), n_host, d_n,
                                                       capacity, ranges, (uint32_t)num_tiles);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

// ---- multi-GPU flow control and the consumer's checksum (include/lcgs_b200.h, peer section) ----------------
__global__ void peer_signal_kernel(uint32_t* flag, uint32_t value)
{
    // kernels of one stream run in order, so every store of the frame has been performed when this kernel starts;
    // the fence orders them (at system scope: the flag may sit in another GPU's memory) before the flag's store
    __threadfence_system();
    asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}

__global__ void peer_wait_kernel(const uint32_t* flag, uint32_t value, long long timeout_cycles, uint32_t* d_timeouts)
{
    const long long t0 = clock64();
    for (;;) {
        uint32_t v;
        asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if ((int32_t)(v - value) >= 0) break;  // sequence numbers: wrap-around safe
        if (clock64() - t0 > timeout_cycles) {
            atomicAdd(d_timeouts, 1u);
            break;
        }
        __nanosleep(500);
    }
    __threadfence_system();
}

__global__ void __launch_bounds__(256) checksum_u32_kernel(const uint4* __restrict__ data, size_t num_vec, const uint32_t* __restrict__ tail,
                                                           uint32_t num_tail, unsigned long long* out)
{
    unsigned long long acc = 0;
    const size_t       stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < num_vec; k += stride) {
        const uint4 v = __ldcs(data + k);  // streamed: read once
        acc += (unsigned long long)v.x + v.y + v.z + v.w;
    }
    if (blockIdx.x == 0 && threadIdx.x < num_tail) acc += tail[threadIdx.x];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, d);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(out, acc);
}

int launch_peer_signal(lcgs_b200_ctx* ctx, uint32_t* flag, uint32_t value, cudaStream_t s)
{
    peer_signal_kernel<<<1, 1, 0, s>>>(flag, value);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_peer_wait(lcgs_b200_ctx* ctx, const uint32_t* flag, uint32_t value, uint32_t timeout_ms, cudaStream_t s)
{
    // clock64 ticks at the SM clock (<= ~2 GHz): 2e6 cycles per millisecond bounds the wait from above
    peer_wait_kernel<<<1, 1, 0, s>>>(flag, value, (long long)timeout_ms * 2000000ll, ctx->d_scalars + LCGS_SCALAR_PEER_TIMEOUTS);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_checksum_u32(lcgs_b200_ctx* ctx, const void* data, size_t num_words, uint64_t* out, cudaStream_t s)
{
    LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(out, 0, sizeof(uint64_t), s));
    if (num_words == 0) return LCGS_B200_OK;
    const size_t num_vec = num_words / 4;
    size_t       blocks  = (num_vec + 255) / 256;
    const size_t max_blocks = (size_t)ctx->num_sms * 4;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks == 0) blocks = 1;
    checksum_u32_kernel<<<(unsigned)blocks, 256, 0, s>>>(reinterpret_cast<const uint4*>(data), num_vec,
                                                         reinterpret_cast<const uint32_t*>(data) + num_vec * 4, (uint32_t)(num_words & 3),
                                                         reinterpret_cast<unsigned long long*>(out));
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

// ---- one clear for everything a fused frame needs zeroed (ClearList, frame_plan.cuh) -----------------------------
__global__ void __launch_bounds__(256) frame_clear_kernel(const __grid_constant__ ClearList cl)
{
    const uint32_t gtid = blockIdx.x * blockDim.x + threadIdx.x, gsize = gridDim.x * blockDim.x;
    for (int r = 0; r < cl.n; r++) {
        uint32_t* const p     = static_cast<uint32_t*>(cl.ptr[r]);
        const uint32_t  words = cl.words[r];
        // 16-byte stores over the aligned middle, 4-byte stores for the (at most three-word) head and tail
        const uint32_t head = (uint32_t)((16u - ((uintptr_t)p & 15u)) & 15u) / 4u;
        const uint32_t h    = head < words ? head : words;
        const uint32_t nvec = (words - h) / 4u;
        uint4* const   v    = reinterpret_cast<uint4*>(p + h);
        for (uint32_t k = gtid; k < nvec; k += gsize) v[k] = make_uint4(0u, 0u, 0u, 0u);
        if (gtid < h) p[gtid] = 0u;
        const uint32_t tail0 = h + nvec * 4u;
        if (gtid < words - tail0) p[tail0 + gtid] = 0u;
    }
}

int launch_clear(lcgs_b200_ctx* ctx, const ClearList& cl, cudaStream_t s)
{
    if (cl.n == 0) return LCGS_B200_OK;
    size_t words = 0;
    for (int r = 0; r < cl.n; r++) words += cl.words[r];
    size_t       blocks     = (words / 4 + 255) / 256;
    const size_t max_blocks = (size_t)ctx->num_sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    if (blocks == 0) blocks = 1;
    frame_clear_kernel<<<(unsigned)blocks, 256, 0, s>>>(cl);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

template <typename T>
static int launch_fill(lcgs_b200_ctx* ctx, T* buf, size_t n, T v, cudaStream_t s)
{
    if (n == 0) return LCGS_B200_OK;
    size_t       blocks     = (n + 1023) / 1024;
    const size_t max_blocks = (size_t)ctx->num_sms * 8;
    if (blocks > max_blocks) blocks = max_blocks;
    fill_kernel<T><<<(unsigned)blocks, 256, 0, s>>>(buf, n, v);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    return LCGS_B200_OK;
}

int launch_fill_u32(lcgs_b200_ctx* ctx, uint32_t* buf, size_t n, uint32_t v, cudaStream_t s) { return launch_fill(ctx, buf, n, v, s); }
int launch_fill_u64(lcgs_b200_ctx* ctx, uint64_t* buf, size_t n, uint64_t v, cudaStream_t s)
{
    return launch_fill(ctx, reinterpret_cast<unsigned long long*>(buf), n, (unsigned long long)v, s);
}
int launch_fill_f32(lcgs_b200_ctx* ctx, float* buf, size_t n, float v, cudaStream_t s) { return launch_fill(ctx, buf, n, v, s); }

}  // namespace lcgs_b200
