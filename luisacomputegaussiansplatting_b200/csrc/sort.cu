// sort.cu -- stage 4: onesweep least-significant-digit radix sort of (uint64 key, uint32 value)
// pairs.  Replaces lcpp DeviceRadixSort<>::SortPairs<ulong,uint> (call site
// lcgs/src/gs_tile_splatter/impl.cpp:134-144), which the reference's README calls crude.
//
// One histogram kernel reads the keys once and counts every digit of every pass (in the fused frame the
// kernels that PRODUCE the keys accumulate the histograms instead); then one "onesweep" kernel per digit
// reads each pair once and writes it once to its final place for that pass: tiles are ranked in shared
// memory per warp (lanes with equal digits found with one ballot per digit bit, or MATCH.ANY for long keys;
// one shared-memory atomic per group), the per-digit global offsets come from a decoupled look-back across
// tiles (a window of predecessors in flight per step), and keys and values are staged through shared memory
// so that global stores are coalesced runs.  The next tile's keys are prefetched into registers behind the
// current tile's look-back and write-out.  Digits are 7 bits wide for the fused frame's tile sort (13 bits =
// 2 passes) and 9 bits otherwise (27-bit depth keys = 3 passes, 45 key bits = 5 passes).
// Stable: ties keep their input order, so equal (tile, depth) keys stay ordered by Gaussian index,
// exactly what the CPU oracle's stable sort yields.
//
// HBM-bound: algorithmic bytes = 8*n (histogram) + 24*n per pass.
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"

namespace lcgs_b200 {

constexpr uint32_t kStatusAggregate = 1u << 30;
constexpr uint32_t kStatusInclusive = 2u << 30;
constexpr uint32_t kStatusValueMask = (1u << 30) - 1u;
constexpr int      kLookbackWindow  = 8;
// onesweep_pass_kernel flags
constexpr int kSweepSkipIfTrivial = 1;

__device__ __forceinline__ uint32_t ld_relaxed_u32(const uint32_t* p)
{
    uint32_t v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ void st_relaxed_u32(uint32_t* p, uint32_t v)
{
    asm volatile("st.relaxed.gpu.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}

__device__ __forceinline__ uint32_t atom_shared_add(uint32_t addr, uint32_t v)
{
    uint32_t old;
    asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(addr), "r"(v) : "memory");
    return old;
}

// 4-byte asynchronous copy global -> shared (LDGSTS): the value never occupies a register
__device__ __forceinline__ void cp_async_u32(uint32_t smem_addr, const uint32_t* gptr)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_addr), "l"(gptr) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory"); }

__device__ __forceinline__ size_t resolve_n(size_t n_host, const uint32_t* d_n, size_t capacity)
{
    if (!d_n) return n_host;
    size_t n = *d_n;
    return n > capacity ? capacity : n;
}

// digit of a 64-bit key: bits [shift, shift+width) -- one funnel shift + one AND
__device__ __forceinline__ uint32_t key_digit(unsigned long long key, int shift, uint32_t mask)
{
    return __funnelshift_r((uint32_t)key, (uint32_t)(key >> 32), shift) & mask;  // shift < 32
}
__device__ __forceinline__ uint32_t key_digit_hi(unsigned long long key, int shift, uint32_t mask)
{
    return ((uint32_t)(key >> 32) >> (shift - 32)) & mask;  // shift >= 32
}

__device__ __forceinline__ uint32_t key_digit(uint32_t key, int shift, uint32_t mask) { return (key >> shift) & mask; }
__device__ __forceinline__ uint32_t key_digit_hi(uint32_t key, int, uint32_t) { return key; }  // unreachable (shift < 32)
__device__ __forceinline__ unsigned long long key_ones(unsigned long long) { return ~0ull; }
__device__ __forceinline__ uint32_t           key_ones(uint32_t) { return ~0u; }

// ---- upfront histogram of every pass's digit ---------------------------------------------------
template <typename KeyT>
__global__ void __launch_bounds__(256)
    radix_histogram_kernel(const KeyT* __restrict__ keys, size_t n_host, const uint32_t* __restrict__ d_n,
                           size_t capacity, uint32_t* __restrict__ hist, const __grid_constant__ SortPassInfo info)
{
    __shared__ uint32_t s_hist[kMaxSortPasses * kMaxRadix];
    const int radix = 1 << info.radix_bits;
    for (int k = threadIdx.x; k < info.num_passes * radix; k += blockDim.x) s_hist[k] = 0u;
    __syncthreads();
    const size_t n      = resolve_n(n_host, d_n, capacity);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const KeyT key = __ldg(keys + k);
#pragma unroll
        for (int p = 0; p < kMaxSortPasses; p++)
            if (p < info.num_passes)
                atomicAdd(&s_hist[(p << info.radix_bits) + (uint32_t)((key >> info.shift[p]) & info.mask[p])], 1u);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < info.num_passes * radix; k += blockDim.x) {
        const uint32_t c = s_hist[k];
        if (c) atomicAdd(hist + k, c);
    }
}

// exclusive scan of one value per thread over a THREADS-thread block
template <int THREADS>
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* s_warp /* [THREADS/32] */)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t  x    = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, x, d);
        if (lane >= d) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    uint32_t pre = 0;
#pragma unroll
    for (int w = 0; w < THREADS / 32; w++)
        if (w < warp) pre += s_warp[w];
    __syncthreads();  // s_warp may be reused
    return pre + x - v;
}

// ---- one onesweep pass -------------------------------------------------------------------------
// THREADS x ITEMS pairs per tile (warp-striped), 2^RBITS digits (one digit per thread, THREADS >=
// 2^RBITS).  Dynamic shared memory:
//   s_keys [TILE]         u64  tile's keys in tile-sorted order
//   s_vals [TILE]         u32  tile's values in tile-sorted order
//   s_wh   [WARPS][RADIX] u32  per-warp digit counters, then each warp's first slot per digit
//   s_base [RADIX]        u32  global position of the digit's first pair minus its first tile slot
template <typename KeyT, int THREADS, int ITEMS, int RBITS>
constexpr size_t sweep_smem_bytes()
{
    return (size_t)THREADS * ITEMS * (sizeof(KeyT) + 4) + (size_t)(THREADS / 32) * (1 << RBITS) * 4 + (size_t)(1 << RBITS) * 4 + (THREADS / 32) * 4 +
           64;
}

// lanes holding the same digit as this lane: MATCH.ANY, or one ballot per digit bit (BITS = RBITS, +1 for
// the "invalid" flag of a partial tile).  MATCH.ANY is the slower of the two on sm_100a (measured on the
// C3 tile sort: 0.368 ms with MATCH, 0.337 ms with 8 ballots per item).
template <int BITS, bool USE_MATCH>
__device__ __forceinline__ unsigned digit_peers(uint32_t d)
{
    if (USE_MATCH) return __match_any_sync(0xFFFFFFFFu, d);
    unsigned peers = 0xFFFFFFFFu;
#pragma unroll
    for (int b = 0; b < BITS; b++) {
        if (BITS <= 9) {
            // peers &= ballot(bit b set) ^ (bit b set ? 0 : ~0), spelled out so that it stays four instructions
            // (test, vote, select, lop3); nvcc otherwise shifts, tests twice and selects per bit
            asm volatile(
                "{\n .reg .pred p;\n .reg .b32 m, s;\n"
                " and.b32 s, %1, %2;\n setp.ne.u32 p, s, 0;\n"
                " vote.sync.ballot.b32 m, p, 0xffffffff;\n"
                " selp.b32 s, 0, 0xffffffff, p;\n"
                " lop3.b32 %0, %0, m, s, 0x60;\n}"
                : "+r"(peers)
                : "r"(d), "r"(1u << b));
        } else {
            // nine or ten bits: ptxas runs out of predicate registers on the spelled-out form
            const bool     bit = (d & (1u << b)) != 0u;
            const unsigned m   = __ballot_sync(0xFFFFFFFFu, bit);
            peers &= m ^ (bit ? 0u : 0xFFFFFFFFu);
        }
    }
    return peers;
}

// HI: the digit lies entirely in the upper 32 bits of a 64-bit key (every pass of the tile sort), so it is a
// shift and a mask of one register; otherwise a funnel shift over both words.
template <typename KeyT, int THREADS, int ITEMS, int RBITS, int MIN_BLOCKS, bool USE_MATCH, bool HI>
__global__ void __launch_bounds__(THREADS, MIN_BLOCKS)
    onesweep_pass_kernel(const KeyT* __restrict__ keys_in, KeyT* __restrict__ keys_out,
                         const uint32_t* __restrict__ vals_in, uint32_t* __restrict__ vals_out, size_t n_host,
                         const uint32_t* __restrict__ d_n, size_t capacity, const uint32_t* __restrict__ hist /* [RADIX] */,
                         uint32_t* status /* [tiles][RADIX] */, uint32_t* ticket, int shift, uint32_t mask,
                         int flags /* kSweep* */)
{
    constexpr int RADIX = 1 << RBITS;
    constexpr int WARPS = THREADS / 32;
    constexpr int TILE  = THREADS * ITEMS;
    static_assert(THREADS >= RADIX && THREADS % 32 == 0, "one thread per digit");
    static_assert((WARPS * RADIX) % THREADS == 0, "counter zeroing");
    static_assert(RADIX % 32 == 0 && THREADS * ITEMS <= 65536, "digit warps are whole warps; tile slots fit 16 bits");

    extern __shared__ __align__(16) unsigned char smem_raw[];
    KeyT* const               s_keys   = reinterpret_cast<KeyT*>(smem_raw);
    uint32_t* const           s_vals   = reinterpret_cast<uint32_t*>(s_keys + TILE);
    uint32_t* const           s_wh     = s_vals + TILE;
    uint32_t* const           s_base   = s_wh + WARPS * RADIX;
    uint32_t* const           s_scan   = s_base + RADIX;  // [WARPS]
    uint32_t* const           s_ticket = s_scan + WARPS;  // [2]

    const int      tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const unsigned lt_mask   = (1u << lane) - 1u;
    const size_t   n         = resolve_n(n_host, d_n, capacity);
    const uint32_t num_tiles = (uint32_t)((n + TILE - 1) / TILE);
    const uint32_t q0        = warp * (ITEMS * 32) + lane;  // warp-striped: item j sits at q0 + 32*j
    const bool     is_digit  = tid < RADIX;
    const uint32_t  s_vals_addr = (uint32_t)__cvta_generic_to_shared(s_vals);
    uint32_t* const my_hist  = s_wh + warp * RADIX;
    const uint32_t  my_hist_addr = (uint32_t)__cvta_generic_to_shared(my_hist);
    // every key has digit 0 in this pass (the top bits of the depth keys): the pass is the identity
    // permutation; the consumers of the sorted list make the same test and read this pass's input
    if ((flags & kSweepSkipIfTrivial) && __ldg(hist) == (uint32_t)n) return;

    auto digit_of = [&](KeyT k) -> uint32_t { return HI ? key_digit_hi(k, shift, mask) : key_digit(k, shift, mask); };
    auto tile_valid = [&](uint32_t t) -> uint32_t {
        const size_t base = (size_t)t * TILE;
        return (uint32_t)((n - base) < (size_t)TILE ? (n - base) : (size_t)TILE);
    };

    // global exclusive scan of this pass's digit histogram (same for every tile)
    const uint32_t bin_base = block_exclusive_scan<THREADS>(is_digit ? __ldg(hist + tid) : 0u, s_scan);

    // Tiles are handed out by a ticket counter.  Every CTA takes its next ticket at the same point of
    // its loop (the top), one tile ahead, so that the keys can be prefetched: tickets then start in
    // (nearly) ticket order, which keeps look-back waits short, and every CTA processes its tickets in
    // increasing order, which keeps the look-back free of deadlock.
    if (tid == 0) s_ticket[0] = atomicAdd(ticket, 1u);
#pragma unroll
    for (int k = 0; k < (WARPS * RADIX) / THREADS; k++) s_wh[tid + k * THREADS] = 0u;
    __syncthreads();
    uint32_t tile = s_ticket[0];

    KeyT key[ITEMS];
    auto load_keys = [&](uint32_t t) {
        if (t >= num_tiles) return;
        const KeyT* src = keys_in + (size_t)t * TILE + q0;
        const uint32_t            nv  = tile_valid(t);
        if (nv == (uint32_t)TILE) {
#pragma unroll
            for (int j = 0; j < ITEMS; j++) key[j] = __ldg(src + 32 * j);
        } else {
#pragma unroll
            for (int j = 0; j < ITEMS; j++) key[j] = (q0 + 32 * j < nv) ? __ldg(src + 32 * j) : key_ones(KeyT());
        }
    };
    load_keys(tile);

    // One tile; `full_c` makes "every slot of the tile holds a pair" a compile-time fact (all tiles but the last),
    // which removes the per-item bounds predicates and the extra ballot for the invalid flag.
    auto process_tile = [&](auto full_c, const uint32_t nvalid) {
        constexpr bool full = decltype(full_c)::value;
        if (tid == 0) s_ticket[1] = atomicAdd(ticket, 1u);  // published by the barrier after ranking

        // ---- rank inside the warp (s_wh is zero on entry): lanes with the same digit are found with
        // match_any; the lowest of them adds the group to the warp's counter with ONE shared-memory atomic
        // and hands the old value to its peers by shuffle.  No register dependency between the items (the
        // same-address atomics of a warp execute in program order), so the 8 chains overlap.
        uint32_t rd[ITEMS];  // (digit << 16) | rank inside (warp, digit); after the scatter: slot in the tile
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const bool     valid  = full || q0 + 32 * j < nvalid;
            const uint32_t d      = valid ? digit_of(key[j]) : (uint32_t)RADIX;
            const unsigned peers  = digit_peers<full ? RBITS : RBITS + 1, USE_MATCH>(d);
            const unsigned lower  = peers & lt_mask;
            uint32_t       before = 0;
            if (valid && lower == 0u) before = atom_shared_add(my_hist_addr + d * 4u, (uint32_t)__popc(peers));
            before = __shfl_sync(0xFFFFFFFFu, before, __ffs(peers) - 1);
            rd[j]  = (d << 16) | (before + __popc(lower));
        }
        __syncthreads();
        const uint32_t next_tile = s_ticket[1];

        // The values never pass through registers: once an item's slot is known (the scatter below), its
        // value is copied global -> shared memory asynchronously (LDGSTS, 4 bytes) straight into that slot,
        // and the copies are waited for behind the look-back.  Holding ITEMS values in registers from here
        // to the scatter made the 256 x 20 geometry spill at its 128-register budget.
        const uint32_t* vsrc = vals_in + (size_t)tile * TILE + q0;

        // ---- per digit (thread d): tile histogram, early publish, first look-back window ---------
        constexpr bool  kCntInRegs = WARPS <= 8 && ITEMS * (int)sizeof(KeyT) < 160;  // otherwise re-read the counters instead of holding them
        uint32_t        tile_count = 0, scan_incl = 0;
        uint32_t        cnt[kCntInRegs ? WARPS : 1];
        uint32_t        st[kLookbackWindow];
        uint32_t* const my_status = status + (size_t)tile * RADIX + tid;
        int             p         = (int)tile - 1;
        if (is_digit) {
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const uint32_t c = s_wh[w * RADIX + tid];
                if (kCntInRegs) cnt[w] = c;
                tile_count += c;
            }
            if (tile > 0) st_relaxed_u32(my_status, kStatusAggregate | tile_count);
            // the predecessors' status words are requested now and consumed after the scatter
#pragma unroll
            for (int k = 0; k < kLookbackWindow; k++)
                st[k] = (p - k >= 0) ? ld_relaxed_u32(status + (size_t)(p - k) * RADIX + tid) : kStatusInclusive;
            // exclusive scan of the digit counts: only the RADIX / 32 digit warps take part
            scan_incl = tile_count;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t y = __shfl_up_sync(0xFFFFFFFFu, scan_incl, d);
                if (lane >= d) scan_incl += y;
            }
            if (lane == 31) s_scan[warp] = scan_incl;
        }
        __syncthreads();
        uint32_t tile_start = 0;
        if (is_digit) {
#pragma unroll
            for (int w = 0; w < RADIX / 32; w++)
                if (w < warp) tile_start += s_scan[w];
            tile_start += scan_incl - tile_count;
            uint32_t run = tile_start;
#pragma unroll
            for (int w = 0; w < WARPS; w++) {
                const uint32_t c      = kCntInRegs ? cnt[w] : s_wh[w * RADIX + tid];
                s_wh[w * RADIX + tid] = run;
                run += c;
            }
        }
        __syncthreads();

        // ---- scatter keys and values into shared memory in tile-sorted order ---------------------
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            if (full || q0 + 32 * j < nvalid) {
                const uint32_t slot = (rd[j] & 0xFFFFu) + my_hist[rd[j] >> 16];
                s_keys[slot] = key[j];
                cp_async_u32(s_vals_addr + slot * 4u, vsrc + 32 * j);
            }
        }
        // this warp's counters are free again: clear them for its next tile (only the warp itself touches
        // them until the barrier after the next ranking)
        __syncwarp();
#pragma unroll
        for (int k = lane; k < RADIX; k += 32) my_hist[k] = 0u;
        // the key registers are free: request the next tile's keys behind the look-back and the write-out
        load_keys(next_tile);

        // ---- decoupled look-back: consume the window requested above, then further windows ---------
        if (is_digit) {
            uint32_t prefix = 0;
            bool     more   = tile > 0;
            while (more) {
#pragma unroll
                for (int k = 0; k < kLookbackWindow; k++) {
                    if (!more) break;
                    if ((st[k] >> 30) == 0u) {  // not published yet: poll again from this tile
                        p -= k;
                        break;
                    }
                    prefix += st[k] & kStatusValueMask;
                    if ((st[k] >> 30) == 2u) more = false;
                    else if (k == kLookbackWindow - 1) p -= kLookbackWindow;
                }
                if (more) {
#pragma unroll
                    for (int k = 0; k < kLookbackWindow; k++)
                        st[k] = (p - k >= 0) ? ld_relaxed_u32(status + (size_t)(p - k) * RADIX + tid) : kStatusInclusive;
                }
            }
            st_relaxed_u32(my_status, kStatusInclusive | ((prefix + tile_count) & kStatusValueMask));
            s_base[tid] = bin_base + prefix - tile_start;
        }
        cp_async_wait_all();  // this thread's value copies have landed; the barrier publishes everybody's
        __syncthreads();

        // ---- coalesced write-out of keys and values ------------------------------------------------
#pragma unroll
        for (int j = 0; j < ITEMS; j++) {
            const uint32_t q = tid + j * THREADS;
            if (full || q < nvalid) {
                const KeyT     k   = s_keys[q];
                const uint32_t dst = s_base[digit_of(k)] + q;
                keys_out[dst]      = k;
                vals_out[dst]      = s_vals[q];
            }
        }
        tile = next_tile;
    };
    while (tile < num_tiles) {
        const uint32_t nvalid = tile_valid(tile);
        if (nvalid == (uint32_t)TILE) process_tile(std::true_type{}, nvalid);
        else process_tile(std::false_type{}, nvalid);
        // s_ticket[1] is rewritten at the next loop top, after every thread has read it (three barriers
        // ago); s_keys / s_vals are rewritten after three more barriers, by which time every thread has
        // finished the loop above; s_scan is rewritten before the next barrier, read before the last one
    }
}

template <typename KeyT>
__global__ void __launch_bounds__(256)
    copy_pairs_kernel(const KeyT* __restrict__ keys_in, KeyT* __restrict__ keys_out,
                      const uint32_t* __restrict__ vals_in, uint32_t* __restrict__ vals_out, size_t n_host,
                      const uint32_t* __restrict__ d_n, size_t capacity)
{
    const size_t n      = resolve_n(n_host, d_n, capacity);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        keys_out[k] = keys_in[k];
        vals_out[k] = vals_in[k];
    }
}

template <typename KeyT>
struct SweepVariant {
    using Kernel = void (*)(const KeyT*, KeyT*, const uint32_t*, uint32_t*, size_t, const uint32_t*, size_t, const uint32_t*,
                            uint32_t*, uint32_t*, int, uint32_t, int);
    Kernel      kernel[2];  // [0] digit anywhere below bit 32 or across it, [1] digit in the upper word (64-bit keys)
    int         threads, tile, radix_bits, blocks_per_sm;
    size_t      smem;
    const char* name;
};
#define LCGS_SWEEP64(T, I, R, B, M)                                                                                         \
    { { onesweep_pass_kernel<unsigned long long, T, I, R, B, M, false>, onesweep_pass_kernel<unsigned long long, T, I, R, B, M, true> }, \
      T, T * I, R, B, sweep_smem_bytes<unsigned long long, T, I, R>(), #T "x" #I " r" #R " " #B "/SM" }
#define LCGS_SWEEP32(T, I, R, B, M)                                                                    \
    { { onesweep_pass_kernel<uint32_t, T, I, R, B, M, false>, onesweep_pass_kernel<uint32_t, T, I, R, B, M, false> }, \
      T, T * I, R, B, sweep_smem_bytes<uint32_t, T, I, R>(), #T "x" #I " r" #R " " #B "/SM" }

// (tile<<32 | depth) instance keys; LCGS_SORT_VARIANT selects another geometry (tuning only).  The geometries
// that lost the sweeps (profiles/README.md) are no longer compiled.
static const SweepVariant<unsigned long long> kSweep64[] = {
    LCGS_SWEEP64(512, 8, 9, 2, true),    // 0: 9-bit digits, MATCH.ANY ranking: long keys (reference flow, 45 bits = 5 passes)
    LCGS_SWEEP64(512, 8, 9, 2, false),   // 1: 9-bit digits, ballot ranking: 15..18 key bits (8K frames)
    LCGS_SWEEP64(256, 20, 7, 2, false),  // 2: 7-bit digits, ballot ranking, 5120-pair tiles: <= 14 key bits (fused flow)
#ifdef LCGS_TUNING
    LCGS_SWEEP64(256, 12, 7, 4, false),  // 3: same, 3072-pair tiles, 4 CTAs/SM
    LCGS_SWEEP64(512, 8, 7, 2, true),    // 4: 7-bit digits, MATCH.ANY ranking (the earlier default)
    LCGS_SWEEP64(256, 16, 7, 3, false),  // 5: 4096-pair tiles, 3 CTAs/SM (85 registers)
    LCGS_SWEEP64(256, 24, 7, 2, false),  // 6: 6144-pair tiles
    LCGS_SWEEP64(384, 14, 7, 2, false),  // 7: 5376-pair tiles, 12 warps per CTA
    LCGS_SWEEP64(512, 10, 7, 2, false),  // 8: 5120-pair tiles, 16 warps per CTA (64 registers)
#endif
};
// 32-bit depth keys of the per-Gaussian sort
static const SweepVariant<uint32_t> kSweep32[] = {
    LCGS_SWEEP32(512, 16, 9, 1, false),  // 0: one 8192-pair tile per SM, ballot ranking
#ifdef LCGS_TUNING
    LCGS_SWEEP32(512, 8, 9, 2, false),   // 1
    LCGS_SWEEP32(512, 8, 9, 2, true),    // 2: MATCH.ANY ranking (the earlier default)
#endif
};
template <typename KeyT>
struct SweepTable;
template <>
struct SweepTable<unsigned long long> {
    static const SweepVariant<unsigned long long>* table() { return kSweep64; }
    static int count() { return (int)(sizeof(kSweep64) / sizeof(kSweep64[0])); }
    static const char* env() { return "LCGS_SORT_VARIANT"; }
};
template <>
struct SweepTable<uint32_t> {
    static const SweepVariant<uint32_t>* table() { return kSweep32; }
    static int count() { return (int)(sizeof(kSweep32) / sizeof(kSweep32[0])); }
    static const char* env() { return "LCGS_SORT32_VARIANT"; }
};

// Geometry used for a sort over `bits` key bits: the environment override (tuning), else 7-bit digits
// when two of them cover the range (the fused frame's 13 tile bits), else 9-bit digits.
template <typename KeyT>
static int sweep_variant_index(int bits)
{
    const int env_idx = LCGS_TUNE_INT(SweepTable<KeyT>::env(), -1);  // -1 outside -DLCGS_TUNING builds
    if (env_idx >= 0 && env_idx < SweepTable<KeyT>::count()) return env_idx;
    // measured: two 7-bit ballot passes for up to 14 tile bits (256 x 20, 2 CTAs/SM); two 9-bit ballot passes up to
    // 18 bits (the 8K frame's 17 tile bits: 4.8 ms vs 5.4 ms with MATCH); MATCH ranking for longer keys
    // (the reference flow's 45 bits = 5 passes: 1.11 ms vs 1.17 ms with ten ballots per item)
    if (sizeof(KeyT) == 8) return bits <= 14 ? 2 : (bits <= 18 ? 1 : 0);
    return 0;                                            // depth keys: 9-bit digits, one 8192-pair tile per SM
}

template <typename KeyT>
int sort_plan_geometry(lcgs_b200_ctx* ctx, size_t bound, int begin_bit, int end_bit, SortPlan<KeyT>* plan)
{
    constexpr int kKeyBits = (int)sizeof(KeyT) * 8;
    LCGS_REQUIRE(ctx, begin_bit >= 0 && end_bit <= kKeyBits && begin_bit <= end_bit, "sort: bad bit range");
    LCGS_REQUIRE(ctx, bound <= (size_t)kStatusValueMask, "sort: more than 2^30-1 pairs");
    const int                 bits  = end_bit - begin_bit;
    const int                 vi    = sweep_variant_index<KeyT>(bits);
    const SweepVariant<KeyT>& var   = SweepTable<KeyT>::table()[vi];
    const int                 rbits = var.radix_bits;
    SortPassInfo&             info  = plan->info;
    info.radix_bits = rbits;
    info.num_passes = (bits + rbits - 1) / rbits;
    LCGS_REQUIRE(ctx, info.num_passes <= kMaxSortPasses, "sort: too many passes");
    for (int p = 0; p < kMaxSortPasses; p++) {
        const int lo  = begin_bit + p * rbits;
        const int w   = (p < info.num_passes) ? ((end_bit - lo) < rbits ? (end_bit - lo) : rbits) : 0;
        info.shift[p] = lo < kKeyBits ? lo : 0;
        info.mask[p]  = w > 0 ? ((1u << w) - 1u) : 0u;
    }
    plan->variant    = vi;
    plan->bound      = bound;
    plan->tiles      = (bound + var.tile - 1) / var.tile;
    plan->hist_ready = false;
    return LCGS_B200_OK;
}
template int sort_plan_geometry<uint32_t>(lcgs_b200_ctx*, size_t, int, int, SortPlan<uint32_t>*);
template int sort_plan_geometry<unsigned long long>(lcgs_b200_ctx*, size_t, int, int, SortPlan<unsigned long long>*);

// in_place: (kin, vals_in) and (kout, vals_out) are both scratch and the passes alternate between them instead of going
// through the workspace (the result is in the output buffers for an odd number of passes, else in the input buffers);
// the last pass returns at once when all its keys have digit 0 (it would be the identity permutation), and *in_place
// receives that pass's input buffers and its histogram, so that the consumer can make the same test (hist[0] == n) and
// read the right pair of buffers.  The other sorts record the profiling events of lcgs_b200_sort_breakdown.
template <typename KeyT>
static int launch_sort_t(lcgs_b200_ctx* ctx, const SortPlan<KeyT>& plan, const KeyT* kin, KeyT* kout, const uint32_t* vals_in,
                         uint32_t* vals_out, size_t n_host, const uint32_t* d_n, size_t capacity, cudaStream_t s,
                         SortedPairsU32* in_place = nullptr)
{
    const size_t bound = plan.bound;
    if (bound == 0) return LCGS_B200_OK;
    const SortPassInfo&       info = plan.info;
    const SweepVariant<KeyT>& var  = SweepTable<KeyT>::table()[plan.variant];
    const unsigned grid_stride_blocks = (unsigned)(((bound + 1023) / 1024) < (size_t)ctx->num_sms * 8
                                                       ? ((bound + 1023) / 1024)
                                                       : (size_t)ctx->num_sms * 8);
    if (info.num_passes == 0) {
        copy_pairs_kernel<KeyT><<<grid_stride_blocks, 256, 0, s>>>(kin, kout, vals_in, vals_out, n_host, d_n, capacity);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
        return LCGS_B200_OK;
    }
    const int    radix = 1 << info.radix_bits;
    const size_t tiles = plan.tiles;

    const bool prof = !in_place && ctx->profiling && ctx->ev_sort[0];
    if (prof) cudaEventRecord(ctx->ev_sort[0], s);
    if (!plan.hist_ready) {
        radix_histogram_kernel<KeyT><<<grid_stride_blocks, 256, 0, s>>>(kin, n_host, d_n, capacity, plan.hist, info);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    }
    if (prof) cudaEventRecord(ctx->ev_sort[1], s);

    // opt in to > 48 KB of dynamic shared memory, once per context (function attributes are per device)
    bool& attr_set = ctx->sweep_attr_set[sizeof(KeyT) == 8 ? 1 : 0][plan.variant];
    if (!attr_set) {
        for (int h = 0; h < 2; h++)
            LCGS_CUDA_CHECK(ctx, cudaFuncSetAttribute(var.kernel[h], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)var.smem));
        attr_set = true;
    }
    const size_t   max_ctas     = (size_t)ctx->num_sms * var.blocks_per_sm;
    const unsigned sweep_blocks = (unsigned)(tiles < max_ctas ? tiles : max_ctas);
    const KeyT*     src_k = kin;
    const uint32_t* src_v = vals_in;
    for (int p = 0; p < info.num_passes; p++) {
        // ping-pong with the workspace so that the last pass lands in (kout, vals_out) and the input survives,
        // or in place (above)
        const bool to_out = in_place ? (p % 2) == 0 : ((info.num_passes - 1 - p) % 2) == 0;
        KeyT*      dst_k  = to_out ? kout : (in_place ? const_cast<KeyT*>(kin) : plan.tmp_keys);
        uint32_t*  dst_v  = to_out ? vals_out : (in_place ? const_cast<uint32_t*>(vals_in) : plan.tmp_vals);
        const bool last = p == info.num_passes - 1;
        if (last && in_place) {
            in_place->alt_keys  = reinterpret_cast<const uint32_t*>(src_k);
            in_place->alt_vals  = src_v;
            in_place->last_hist = plan.hist + (size_t)p * radix;
        }
        const int hi = (sizeof(KeyT) == 8 && info.shift[p] >= 32) ? 1 : 0;
        var.kernel[hi]<<<sweep_blocks, var.threads, var.smem, s>>>(src_k, dst_k, src_v, dst_v, n_host, d_n, capacity,
                                                              plan.hist + (size_t)p * radix,
                                                              plan.status + (size_t)p * tiles * radix, plan.ticket + p,
                                                              info.shift[p], info.mask[p],
                                                              (last && in_place) ? kSweepSkipIfTrivial : 0);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
        src_k = dst_k;
        src_v = dst_v;
    }
    if (prof) {
        cudaEventRecord(ctx->ev_sort[2], s);
        ctx->sort_passes   = info.num_passes;
        ctx->ev_sort_valid = 1;
    }
    return LCGS_B200_OK;
}

int launch_sort(lcgs_b200_ctx* ctx, const uint64_t* keys_in, uint64_t* keys_out, const uint32_t* vals_in,
                uint32_t* vals_out, size_t n_host, const uint32_t* d_n, size_t capacity, int begin_bit, int end_bit,
                cudaStream_t s)
{
    const size_t bound = d_n ? capacity : n_host;
    if (bound == 0) return LCGS_B200_OK;
    if (!d_n) capacity = n_host;
    SortPlan<unsigned long long> plan;
    int rc = sort_plan_geometry<unsigned long long>(ctx, bound, begin_bit, end_bit, &plan);
    if (rc) return rc;
    plan.ticket = ctx->d_scalars + LCGS_SCALAR_SORT_TICKET;
    const SortPassInfo& info = plan.info;
    if (info.num_passes > 0) {
        const SortWsLayout l = sort_ws_layout(bound, sort_status_bound(bound));
        if ((rc = ws_reserve(ctx, ctx->sort_ws, l.bytes))) return rc;
        char* ws      = (char*)ctx->sort_ws.ptr;
        plan.hist     = (uint32_t*)(ws + kHistSlotBytes);
        plan.status   = (uint32_t*)(ws + l.status);
        plan.tmp_keys = (unsigned long long*)(ws + l.keys);
        plan.tmp_vals = (uint32_t*)(ws + l.vals);
        // zero this sort's histograms + the look-back status (contiguous) and the tickets
        LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(plan.hist, 0, (size_t)((char*)plan.status - (char*)plan.hist) + sort_status_bytes(plan), s));
        LCGS_CUDA_CHECK(ctx, cudaMemsetAsync(plan.ticket, 0, kMaxSortPasses * sizeof(uint32_t), s));
    }
    return launch_sort_t<unsigned long long>(ctx, plan, reinterpret_cast<const unsigned long long*>(keys_in),
                                             reinterpret_cast<unsigned long long*>(keys_out), vals_in, vals_out, n_host, d_n,
                                             capacity, s);
}

// ---- fused frame: the kernel that PRODUCES the keys also accumulates the digit histograms (FramePlan) -------------
int sort_run_u32(lcgs_b200_ctx* ctx, const SortPlan<uint32_t>& plan, uint32_t* keys_a, uint32_t* keys_b, uint32_t* vals_a,
                 uint32_t* vals_b, const uint32_t* d_n, size_t capacity, SortedPairsU32* res, cudaStream_t s)
{
    const bool in_b = (plan.info.num_passes % 2) == 1;  // pass p writes b for even p, a for odd p
    res->keys = res->alt_keys = in_b ? keys_b : keys_a;
    res->vals = res->alt_vals = in_b ? vals_b : vals_a;
    res->last_hist = nullptr;
    if (plan.info.num_passes == 0) return LCGS_B200_OK;  // nothing to sort by: the input is the result
    return launch_sort_t<uint32_t>(ctx, plan, keys_a, keys_b, vals_a, vals_b, 0, d_n, capacity, s, res);
}

int sort_run_u64(lcgs_b200_ctx* ctx, const SortPlan<unsigned long long>& plan, const uint64_t* keys_in, uint64_t* keys_out,
                 const uint32_t* vals_in, uint32_t* vals_out, const uint32_t* d_n, size_t capacity, cudaStream_t s)
{
    return launch_sort_t<unsigned long long>(ctx, plan, reinterpret_cast<const unsigned long long*>(keys_in),
                                             reinterpret_cast<unsigned long long*>(keys_out), vals_in, vals_out, 0, d_n, capacity, s);
}

}  // namespace lcgs_b200
