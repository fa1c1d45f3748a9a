// frame_plan.cuh -- where the scratch of a depth-ordered ("fused") frame lives.  The stage constants that size it, the
// layouts of the scan, sort and emission workspaces, the device-scalar words, and place_frame(), which carves one frame's
// regions out of the workspaces reserve_all (capi.cu) reserved from the same layout functions.  Plain arithmetic on sizes
// and base pointers, no context and no CUDA call: tests/test_frame_plan_cpu.py compiles this header with g++.
#pragma once

#include <stddef.h>
#include <stdint.h>
#include <vector_types.h>

// Device scalars (lcgs_b200_ctx::d_scalars), 32-bit words.
#define LCGS_SCALAR_NUM_RENDERED  0
#define LCGS_SCALAR_NUM_TOUCHING  1   /* Gaussians with tiles_touched > 0 (fused path) */
#define LCGS_SCALAR_SCAN_TICKET   2
#define LCGS_SCALAR_SORT_TICKET   3   /* .. 3 + kMaxSortPasses - 1, one per pass; fused frame: depth sort + 0..3, tile sort + 4..7 */
#define LCGS_SCALAR_OVERFLOW      13  /* 1 iff the last frame's num_rendered exceeded its list_capacity (device-side test) */
#define LCGS_SCALAR_CAPACITY      14  /* that frame's list_capacity (clamped to 2^32-1), written in-stream; = OVERFLOW + 1 */
#define LCGS_SCALAR_PEER_TIMEOUTS 15  /* sticky: peer waits that gave up (lcgs_b200_peer_error) */
#define LCGS_SCALAR_DUP_TICKET    16  /* the emission's ticket */
#define LCGS_SCALAR_BIG_COUNTERS  17  /* + 18: entry / piece counters of the emission's big-Gaussian lists */
#define LCGS_NUM_SCALARS          24

namespace lcgs_b200 {

struct Workspace {
    void*  ptr   = nullptr;
    size_t bytes = 0;
};

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// ---- scan (scan.cu) --------------------------------------------------------------------------------------------------
constexpr int kScanThreads       = 256;
constexpr int kScanItems         = 16;
constexpr int kScanTile          = kScanThreads * kScanItems;
constexpr int kCompactItems      = 8;                            // scan_compact_kernel: Gaussians per thread
constexpr int kCompactTile       = kScanThreads * kCompactItems;  // 2048 Gaussians per tile
constexpr int kCompactHistPasses = 4;                            // digit passes scan_compact_kernel can count

// ---- instance emission (binning.cu) ----------------------------------------------------------------------------------
constexpr int      kEmitThreads    = 256;
constexpr int      kEmitItems      = 4;  // Gaussians per thread and tile: chunk c of a warp is 32 consecutive ones
constexpr int      kEmitTile       = kEmitThreads * kEmitItems;
constexpr int      kEmitHistPasses = 2;     // digit passes the emission kernels can count
constexpr uint32_t kBigPiece       = 2048;  // instances of a big Gaussian per emit_big_kernel CTA
constexpr uint32_t kBigThreshold   = 128;   // a Gaussian over this many tiles is big
struct BigEntry {
    uint32_t dst, cnt, xy0, w, dbits, idx, pad0, pad1;  // first output slot, tile count, x0 | y0<<16, rect width, depth bits, Gaussian
};
struct BigLists {
    BigEntry* entries;
    uint2*    pieces;    // (entry, piece index)
    uint32_t* counters;  // [0] entries, [1] pieces
    uint32_t  entry_capacity, piece_capacity, threshold;
};

// emit_ws: [entries][pieces].  Each big Gaussian holds more than `threshold` instances, so a frame within its list
// capacity has at most capacity / (threshold + 1) of them (a frame that overflows is reported as such; entries beyond
// are dropped).
struct EmitWsLayout {
    uint32_t entry_capacity, piece_capacity;
    size_t   pieces, bytes;
};
inline EmitWsLayout emit_ws_layout(int P, size_t capacity, uint32_t threshold)
{
    EmitWsLayout l;
    const size_t by_p = (size_t)(P > 0 ? P : 1), by_cap = capacity / ((size_t)threshold + 1) + 1;
    l.entry_capacity  = (uint32_t)(by_p < by_cap ? by_p : by_cap);
    l.piece_capacity  = (uint32_t)(capacity / kBigPiece + l.entry_capacity + 1);
    l.pieces          = (size_t)l.entry_capacity * sizeof(BigEntry);
    l.bytes           = l.pieces + (size_t)l.piece_capacity * sizeof(uint2);
    return l;
}

// scan_ws of a fused frame, one 64-bit look-back status word per tile: [scan sum chain][scan count chain][emission chain]
inline size_t compact_tiles(int P) { return ((size_t)(P > 0 ? P : 1) + kCompactTile - 1) / kCompactTile; }
inline size_t emit_tiles(int P) { return ((size_t)(P > 0 ? P : 1) + kEmitTile - 1) / kEmitTile; }
inline size_t frame_scan_ws_bytes(int P) { return (2 * compact_tiles(P) + emit_tiles(P)) * sizeof(unsigned long long); }

// ---- radix sort (sort.cu) --------------------------------------------------------------------------------------------
constexpr int    kMaxSortPasses   = 8;  // 64 key bits in 9-bit digits
constexpr int    kMaxRadixBits    = 9;
constexpr int    kMaxRadix        = 1 << kMaxRadixBits;
constexpr int    kMinSweepTile    = 2048;  // no sweep variant has smaller tiles
constexpr size_t kHistSlotBytes   = (size_t)kMaxSortPasses * kMaxRadix * sizeof(uint32_t);  // 16 KB, 256-byte multiple
constexpr int    kFrameSortPasses = 4;  // each sort of a fused frame: four tickets

struct SortPassInfo {
    int      num_passes;
    int      radix_bits;
    int      shift[kMaxSortPasses];
    uint32_t mask[kMaxSortPasses];
};

// digit layout of a sort, for kernels that accumulate its histograms while producing the keys
struct SortDigits {
    uint32_t* hist;  // [num_passes][1 << radix_bits], zeroed
    int       num_passes, radix_bits;
    int       shift[kMaxSortPasses];
    uint32_t  mask[kMaxSortPasses];
};

// One sort: geometry from sort_plan_geometry (sort.cu), memory and ticket from its caller.
template <typename KeyT>
struct SortPlan {
    SortPassInfo info;
    int          variant;
    size_t       bound, tiles;
    uint32_t *   hist = nullptr, *status = nullptr, *tmp_vals = nullptr, *ticket = nullptr;
    KeyT*        tmp_keys   = nullptr;
    bool         hist_ready = false;  // the kernel that produces the keys fills `hist`: the sort runs no histogram kernel
};

// look-back status of one sort: [pass][tile][1 << radix_bits] u32
template <typename KeyT>
inline size_t sort_status_bytes(const SortPlan<KeyT>& p)
{
    return (size_t)p.info.num_passes * p.tiles * ((size_t)1 << p.info.radix_bits) * sizeof(uint32_t);
}

// Digits for the producer of a sort's keys: all zero (no histogram) unless the producer fills the histograms.
template <typename KeyT>
inline SortDigits producer_digits(const SortPlan<KeyT>& p)
{
    SortDigits d{};
    if (!p.hist_ready) return d;
    d.hist       = p.hist;
    d.num_passes = p.info.num_passes;
    d.radix_bits = p.info.radix_bits;
    for (int k = 0; k < kMaxSortPasses; k++) { d.shift[k] = p.info.shift[k]; d.mask[k] = p.info.mask[k]; }
    return d;
}

// sort_ws: [hist slot 0][hist slot 1][look-back status][tmp keys: n x 8 B][tmp vals: n x 4 B], regions 256-byte aligned.
// The depth sort of a fused frame uses hist slot 0, every other sort slot 1: the consumers of the depth-sorted list still
// read the depth sort's last histogram (to learn whether its last pass skipped itself) after the tile sort has started.
struct SortWsLayout {
    size_t status, keys, vals, bytes;
};
inline SortWsLayout sort_ws_layout(size_t n, size_t status_bytes)
{
    SortWsLayout l;
    l.status = 2 * kHistSlotBytes;
    l.keys   = align256(l.status + status_bytes);
    l.vals   = align256(l.keys + n * sizeof(uint64_t));
    l.bytes  = align256(l.vals + n * sizeof(uint32_t));
    return l;
}
// any sort of up to n pairs: kMaxSortPasses passes of kMaxRadix digits over tiles of kMinSweepTile pairs
inline size_t sort_status_bound(size_t n) { return (size_t)kMaxSortPasses * ((n + kMinSweepTile - 1) / kMinSweepTile) * kMaxRadix * sizeof(uint32_t); }
inline size_t sort_temp_bytes(size_t n) { return sort_ws_layout(n, sort_status_bound(n)).bytes; }

// ---- one kernel clears a fused frame's scratch (frame_clear_kernel, binning.cu) ---------------------------------------
// (nine cudaMemsetAsync nodes per frame cost ~25 us of a 1.5 ms frame)
struct ClearList {
    static constexpr int kMax = 8;
    void*    ptr[kMax];
    uint32_t words[kMax];  // 32-bit words; ptr 4-byte aligned
    int      n = 0;
};
struct ClearRegion {
    void*  ptr;
    size_t bytes;
};
// Regions of zero bytes are left out; a list of more than ClearList::kMax regions does not compile.
template <int N>
inline ClearList make_clear_list(const ClearRegion (&r)[N])
{
    static_assert(N <= ClearList::kMax, "one clear kernel takes at most ClearList::kMax regions");
    ClearList cl;
    for (int i = 0; i < N; i++) {
        if (r[i].bytes == 0) continue;
        cl.ptr[cl.n]   = r[i].ptr;
        cl.words[cl.n] = (uint32_t)((r[i].bytes + 3) / 4);
        cl.n++;
    }
    return cl;
}

// ---- the frame plan --------------------------------------------------------------------------------------------------
// Everything the tail of a fused frame (scan+compaction -> depth sort -> emission -> tile sort) reads and writes
// besides the caller's buffers, placed before its first kernel so that ONE kernel zeroes all of it.
struct FramePlan {
    SortPlan<uint32_t>           depth;  // the touching Gaussians by depth: <= P pairs, 32 key bits
    SortPlan<unsigned long long> tile;   // the instances by tile, stable: <= L pairs, key bits [32, end_bit)
    unsigned long long *scan_sum, *scan_count, *emit_status;  // look-back chains
    uint32_t *          scan_ticket, *emit_ticket;
    BigLists            big;
    ClearList           clear;
};

// Places one fused frame in the workspaces reserved for it.  `fp->depth` and `fp->tile` carry their geometry on entry.
// Returns nullptr, or why the frame does not fit: a frame never grows a workspace, because growing synchronises the
// device and breaks graph capture.
inline const char* place_frame(FramePlan* fp, int P, size_t L, uint32_t big_threshold, const Workspace& scan_ws,
                               const Workspace& sort_ws, const Workspace& emit_ws, uint32_t* scalars, uint32_t* ranges,
                               size_t num_tiles)
{
    SortPlan<uint32_t>&           d = fp->depth;
    SortPlan<unsigned long long>& t = fp->tile;
    if (d.info.num_passes > kFrameSortPasses || t.info.num_passes > kFrameSortPasses)
        return "sort: a fused frame's sorts have at most four passes each";

    // sort_ws: both sorts' status words back to back; the depth sort ping-pongs between its caller's two buffers
    const size_t       s32 = align256(sort_status_bytes(d)), s64 = align256(sort_status_bytes(t));
    const SortWsLayout sl  = sort_ws_layout(L, s32 + s64);
    if (sl.bytes > sort_ws.bytes) return "frame plan: sort workspace smaller than the frame's layout";
    char* const sw = (char*)sort_ws.ptr;
    d.hist         = (uint32_t*)sw;
    d.status       = (uint32_t*)(sw + sl.status);
    d.tmp_keys     = nullptr;
    d.tmp_vals     = nullptr;
    d.ticket       = scalars + LCGS_SCALAR_SORT_TICKET;
    t.hist         = (uint32_t*)(sw + kHistSlotBytes);
    t.status       = (uint32_t*)(sw + sl.status + s32);
    t.tmp_keys     = (unsigned long long*)(sw + sl.keys);
    t.tmp_vals     = (uint32_t*)(sw + sl.vals);
    t.ticket       = scalars + LCGS_SCALAR_SORT_TICKET + kFrameSortPasses;
    // the compaction counts the depth digits, the emission the tile digits (in the upper key word, at most two passes)
    d.hist_ready = s32 > 0 && d.info.num_passes <= kCompactHistPasses && d.info.radix_bits <= kMaxRadixBits;
    t.hist_ready = s64 > 0 && t.info.num_passes >= 1 && t.info.num_passes <= kEmitHistPasses &&
                   t.info.radix_bits <= kMaxRadixBits && t.info.shift[0] >= 32;

    const size_t scan_bytes = frame_scan_ws_bytes(P);
    if (scan_bytes > scan_ws.bytes) return "frame plan: scan workspace smaller than the frame's layout";
    fp->scan_sum    = (unsigned long long*)scan_ws.ptr;
    fp->scan_count  = fp->scan_sum + compact_tiles(P);
    fp->emit_status = fp->scan_sum + 2 * compact_tiles(P);
    fp->scan_ticket = scalars + LCGS_SCALAR_SCAN_TICKET;
    fp->emit_ticket = scalars + LCGS_SCALAR_DUP_TICKET;

    const EmitWsLayout el = emit_ws_layout(P, L, big_threshold);
    if (el.bytes > emit_ws.bytes) return "frame plan: emission workspace smaller than the frame's layout";
    fp->big = BigLists{ (BigEntry*)emit_ws.ptr, (uint2*)((char*)emit_ws.ptr + el.pieces), scalars + LCGS_SCALAR_BIG_COUNTERS,
                        el.entry_capacity, el.piece_capacity, big_threshold };

    const ClearRegion regions[] = {
        { sw, sl.status + s32 + s64 },  // both histogram slots, both sorts' status
        { scan_ws.ptr, scan_bytes },
        { scalars + LCGS_SCALAR_SCAN_TICKET, 10 * sizeof(uint32_t) },  // scan ticket, 8 sort tickets, one spare word
        { scalars + LCGS_SCALAR_DUP_TICKET, 3 * sizeof(uint32_t) },    // emission ticket, big-list counters
        { ranges, num_tiles * 2 * sizeof(uint32_t) },
    };
    fp->clear = make_clear_list(regions);
    return nullptr;
}

// What reserve_all reserves for frames of up to P >= 1 Gaussians and L instances.  Every frame place_frame accepts fits:
// its two sorts have at most four passes each, over tiles of at least kMinSweepTile pairs, so their status words stay
// within sort_status_bound.
struct FrameWsBytes {
    size_t scan, sort, emit;
};
inline FrameWsBytes frame_ws_bytes(int P, size_t L, uint32_t big_threshold)
{
    return { frame_scan_ws_bytes(P), sort_temp_bytes(L > (size_t)P ? L : (size_t)P), emit_ws_layout(P, L, big_threshold).bytes };
}

}  // namespace lcgs_b200
