// Host build of the fused frame's plan (csrc/frame_plan.cuh) for tests/test_frame_plan_cpu.py: place_frame() over fake
// workspaces of exactly the size reserve_all reserves, with every region reported back.  Test-only code.
#include "../../luisacomputegaussiansplatting_b200/csrc/frame_plan.cuh"

using namespace lcgs_b200;

#define FP_API extern "C" __attribute__((visibility("default")))

// Fake device addresses: region space w starts at w << 40 (1 scan_ws, 2 sort_ws, 3 emit_ws, 4 device scalars, 5 ranges).
static char* space(int w) { return (char*)((uintptr_t)w << 40); }

struct Region {
    uint64_t addr, bytes, align;
    int      zeroed;  // must be zero when the frame's first kernel starts
};

// geom = { passes, radix_bits, tile } of the depth sort, then of the tile sort.  Returns 0 and fills `out`, `clear` and
// `reserved` (scan, sort, emit bytes) if the frame fits, 1 if place_frame refused it.
FP_API int fp_plan(int P, uint64_t L, uint64_t num_tiles, const int* geom, uint64_t* reserved, Region* out, int* n_out,
                   uint64_t* clear, int* n_clear)
{
    const FrameWsBytes r = frame_ws_bytes(P > 0 ? P : 1, L, kBigThreshold);  // reserve_all(ctx, P > 0 ? P : 1, L)
    reserved[0] = r.scan; reserved[1] = r.sort; reserved[2] = r.emit;
    Workspace scan_ws, sort_ws, emit_ws;
    scan_ws.ptr = space(1); scan_ws.bytes = r.scan;
    sort_ws.ptr = space(2); sort_ws.bytes = r.sort;
    emit_ws.ptr = space(3); emit_ws.bytes = r.emit;
    uint32_t* const scalars = (uint32_t*)space(4);

    FramePlan fp;
    const size_t bound[2] = { (size_t)(P > 0 ? P : 0), L };
    SortPassInfo* info[2] = { &fp.depth.info, &fp.tile.info };
    size_t*       tiles[2] = { &fp.depth.tiles, &fp.tile.tiles };
    for (int k = 0; k < 2; k++) {
        info[k]->num_passes = geom[3 * k];
        info[k]->radix_bits = geom[3 * k + 1];
        info[k]->shift[0]   = k == 0 ? 0 : 32;
        *tiles[k]           = (bound[k] + geom[3 * k + 2] - 1) / geom[3 * k + 2];
    }
    fp.depth.bound = bound[0];
    fp.tile.bound  = bound[1];
    if (place_frame(&fp, P, L, kBigThreshold, scan_ws, sort_ws, emit_ws, scalars, (uint32_t*)space(5), num_tiles)) return 1;

    int  n   = 0;
    auto add = [&](const void* p, uint64_t bytes, uint64_t align, int zeroed) {
        if (bytes) out[n++] = Region{ (uint64_t)(uintptr_t)p, bytes, align, zeroed };
    };
    const SortPlan<uint32_t>&           d = fp.depth;
    const SortPlan<unsigned long long>& t = fp.tile;
    if (d.bound) {
        add(d.hist, (uint64_t)d.info.num_passes << d.info.radix_bits << 2, 4, 1);
        add(d.status, sort_status_bytes(d), 4, 1);
        add(d.ticket, 4 * d.info.num_passes, 4, 1);
    }
    if (t.bound) {
        add(t.hist, (uint64_t)t.info.num_passes << t.info.radix_bits << 2, 4, 1);
        add(t.status, sort_status_bytes(t), 4, 1);
        add(t.ticket, 4 * t.info.num_passes, 4, 1);
        add(t.tmp_keys, 8 * L, 8, 0);
        add(t.tmp_vals, 4 * L, 4, 0);
    }
    add(fp.scan_sum, 8 * compact_tiles(P), 8, 1);
    add(fp.scan_count, 8 * compact_tiles(P), 8, 1);
    add(fp.emit_status, 8 * emit_tiles(P), 8, 1);
    add(fp.scan_ticket, 4, 4, 1);
    add(fp.emit_ticket, 4, 4, 1);
    add(fp.big.counters, 8, 4, 1);
    add(fp.big.entries, (uint64_t)fp.big.entry_capacity * sizeof(BigEntry), 4, 0);
    add(fp.big.pieces, (uint64_t)fp.big.piece_capacity * 8, 8, 0);
    add(space(5), 8 * num_tiles, 4, 1);  // the frame's ranges
    *n_out = n;
    for (int k = 0; k < fp.clear.n; k++) {
        clear[2 * k]     = (uint64_t)(uintptr_t)fp.clear.ptr[k];
        clear[2 * k + 1] = 4ull * fp.clear.words[k];
    }
    *n_clear = fp.clear.n;
    return 0;
}

// Scalar words that hold results across frames: no ticket may use them and the frame's clear must leave them alone.
FP_API void fp_result_scalars(int* w)
{
    w[0] = LCGS_SCALAR_NUM_RENDERED; w[1] = LCGS_SCALAR_NUM_TOUCHING; w[2] = LCGS_SCALAR_OVERFLOW;
    w[3] = LCGS_SCALAR_CAPACITY; w[4] = LCGS_SCALAR_PEER_TIMEOUTS; w[5] = LCGS_NUM_SCALARS;
}
