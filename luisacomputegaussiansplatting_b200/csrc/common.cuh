// common.cuh -- context, workspace and launch helpers shared by the stage kernels.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/lcgs_b200.h"
#include "frame_plan.cuh"
#include "lcgs_math.cuh"

namespace lcgs_b200 {

constexpr int kNumSMs = 148;  // B200; the real count is queried at ctx creation

// Per-Gaussian record the blend kernel gathers: three float4 (48 B, two 32-B sectors).
//   r0 = (pix.x, pix.y, -0.5*conic.x, -conic.y)
//   r1 = (-0.5*conic.z, power threshold of the alpha test, log2(opacity), cull quotient ry or NaN)
//   r2 = (red, green, blue, cull quotient rx)            -- see cull_coef() in lcgs_math.cuh
constexpr int kRecordFloat4s = 3;

// (thr, l2op) = (alpha_threshold(opacity), log2f(opacity)): the two per-Gaussian constants of the alpha test.
// Written by the forward's preprocess and by build_records_kernel (preprocess.cu), which also rebuilds them for the
// backward from the frame's buffers.
__device__ __forceinline__ void write_record(float4* rec, const Splat2D& s, float thr, float l2op, const float* rgb)
{
    const float    a = -0.5f * s.conic[0], b = -s.conic[1], c = -0.5f * s.conic[2];
    const CullCoef k = cull_coef(s.px, s.py, a, b, c, thr);
    rec[0] = make_float4(s.px, s.py, a, b);
    rec[1] = make_float4(c, thr, l2op, k.ry);  // the blend evaluates alpha as 2^(power*log2e + log2(opacity))
    rec[2] = make_float4(rgb[0], rgb[1], rgb[2], k.rx);
}

// Depth keys of the per-Gaussian sort are stored relative to the bit pattern of 0.2f, the smallest
// depth a Gaussian that touches a tile can have (near cull, gs_projector/shader.cpp:121): for
// depth < 0.2 * 2^16 they fit in 27 bits = three 9-bit digits, and the fourth pass skips itself.
constexpr uint32_t kDepthKeyBase = 0x3E4CCCCDu;

}  // namespace lcgs_b200

// The opaque context of the C ABI.
struct lcgs_b200_ctx {
    int          device     = 0;
    int          num_sms    = lcgs_b200::kNumSMs;
    char         last_error[256];
    uint32_t*    d_scalars  = nullptr;  // LCGS_SCALAR_* (frame_plan.cuh)
    uint32_t*    h_scalars  = nullptr;  // pinned mirror
    // workspaces, grown geometrically and never shrunk (like ensure_*_temp_buffer,
    // lcgs/src/gs_tile_splatter/impl.cpp:31-61)
    lcgs_b200::Workspace scan_ws;     // look-back tile status
    lcgs_b200::Workspace sort_ws;     // histograms + look-back status + ping-pong pair buffer
    lcgs_b200::Workspace record_ws;   // packed per-Gaussian blend records
    lcgs_b200::Workspace order_ws;    // fused path: packed rects + compacted/sorted (depth, index) pairs + offsets
    lcgs_b200::Workspace tile_order_ws;  // blend: tile ids, longest list first
    lcgs_b200::Workspace emit_ws;        // emission: entries + pieces of the Gaussians expanded by emit_big_kernel
    lcgs_b200::Workspace grad_ws;        // backward: packed per-Gaussian gradient of the blend's inputs [P][12]
    // per-stage timing
    int          profiling  = 0;
    cudaEvent_t  ev[16];
    int          ev_count   = 0;
    int          ev_valid   = 0;
    bool         sweep_attr_set[2][32] = {};  // onesweep variants whose shared-memory opt-in has been done
    cudaEvent_t  ev_sort[3] = { nullptr, nullptr, nullptr };  // before histogram, before passes, after passes
    int          sort_passes = 0;
    int          ev_sort_valid = 0;
};

#define LCGS_CUDA_CHECK(ctx, expr)                                                                   \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            if (ctx)                                                                                 \
                snprintf((ctx)->last_error, sizeof((ctx)->last_error), "%s:%d: %s: %s", __FILE__,    \
                         __LINE__, #expr, cudaGetErrorString(e__));                                  \
            return LCGS_B200_ERR_CUDA;                                                               \
        }                                                                                            \
    } while (0)

#define LCGS_REQUIRE(ctx, cond, msg)                                                                 \
    do {                                                                                             \
        if (!(cond)) {                                                                               \
            if (ctx) snprintf((ctx)->last_error, sizeof((ctx)->last_error), "%s", msg);              \
            return LCGS_B200_ERR_INVALID;                                                            \
        }                                                                                            \
    } while (0)

namespace lcgs_b200 {

int ws_reserve(lcgs_b200_ctx* ctx, Workspace& ws, size_t bytes);

// Geometry overrides by environment variable exist only in -DLCGS_TUNING builds (build.py --tuning, a separate
// library used by scripts/tune_*.py); the production library always runs the measured defaults.
#ifdef LCGS_TUNING
int tuning_env_int(const char* name, int fallback);
#define LCGS_TUNE_INT(name, fallback) ::lcgs_b200::tuning_env_int(name, fallback)
#else
#define LCGS_TUNE_INT(name, fallback) (fallback)
#endif

int launch_clear(lcgs_b200_ctx* ctx, const ClearList& cl, cudaStream_t s);

// stage launchers (one group per .cu); all enqueue on `s` and return an lcgs_b200_status
int launch_preprocess_fused(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                            const lcgs_b200_frame* fr, float4* records, uint2* rects, cudaStream_t s);
// the fused frame's stages take their scratch, tickets and histograms from its plan (frame_plan.cuh)
int launch_scan_compact(lcgs_b200_ctx* ctx, const uint32_t* tiles_touched, const float* depth, int P, uint32_t* offsets,
                        uint32_t* ckeys, uint32_t* cvals, uint32_t* d_total, uint32_t* d_count, const FramePlan& fp,
                        cudaStream_t s);
// Where a u32 sort left its result: (keys, vals), or (alt_keys, alt_vals) when the last pass found all
// its keys in digit 0 and skipped itself -- the case iff last_hist && *last_hist == n (device-side test).
struct SortedPairsU32 {
    const uint32_t *keys, *vals, *alt_keys, *alt_vals, *last_hist;
};
__device__ __forceinline__ bool sorted_in_alt(const SortedPairsU32& r, uint32_t n) { return r.last_hist && __ldg(r.last_hist) == n; }
int launch_duplicate_keys_sorted(lcgs_b200_ctx* ctx, const uint32_t* d_m, int P, int W, int H, int num_rows,
                                 const SortedPairsU32& sorted, const uint2* rects, uint64_t* keys, uint32_t* vals,
                                 size_t capacity, int row0, const FramePlan& fp, cudaStream_t s);
// digit cut, kernel geometry and tile count of a sort over `bound` pairs; no memory, no ticket
template <typename KeyT>
int sort_plan_geometry(lcgs_b200_ctx* ctx, size_t bound, int begin_bit, int end_bit, SortPlan<KeyT>* plan);
// Sorts (keys_a, vals_a) using (keys_b, vals_b) as the ping-pong partner; both pairs are scratch.  The
// result is in res->keys/vals, or in res->alt_* when the last pass skipped itself (SortedPairsU32).
int sort_run_u32(lcgs_b200_ctx* ctx, const SortPlan<uint32_t>& plan, uint32_t* keys_a, uint32_t* keys_b, uint32_t* vals_a,
                 uint32_t* vals_b, const uint32_t* d_n, size_t capacity, SortedPairsU32* res, cudaStream_t s);
int sort_run_u64(lcgs_b200_ctx* ctx, const SortPlan<unsigned long long>& plan, const uint64_t* keys_in, uint64_t* keys_out,
                 const uint32_t* vals_in, uint32_t* vals_out, const uint32_t* d_n, size_t capacity, cudaStream_t s);
int launch_sh(lcgs_b200_ctx* ctx, int P, int deg, const float* cam_pos, const float* pos, const float* sh, float* color,
              cudaStream_t s);
int launch_project(lcgs_b200_ctx* ctx, int P, const float* pos, const float* scale, const float* rotq,
                   float scale_modifier, const ViewParams& vp, float* means_2d, float* depth, float* covs_2d,
                   cudaStream_t s);
int launch_allocate_tiles(lcgs_b200_ctx* ctx, int P, int W, int H, const float* depth, float* means_2d, float* covs_2d,
                          uint32_t* tiles_touched, int32_t* radii, int row0, int row1, cudaStream_t s);
// alpha_consts (lcgs_b200_scene_prepare) and tiles_touched may be null
int launch_build_records(lcgs_b200_ctx* ctx, int P, const float* means_2d, const float* conic, const float* opacity,
                         const float* alpha_consts, const float* color, const uint32_t* tiles_touched, float4* records,
                         cudaStream_t s);
int launch_scan(lcgs_b200_ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, uint32_t* d_total, cudaStream_t s);
int launch_duplicate_keys(lcgs_b200_ctx* ctx, int P, int W, int H, const float* means_2d, const uint32_t* offsets,
                          const int32_t* radii, const float* depth, uint64_t* keys, uint32_t* vals, size_t capacity,
                          int row0, int row1, cudaStream_t s);
int launch_sort(lcgs_b200_ctx* ctx, const uint64_t* keys_in, uint64_t* keys_out, const uint32_t* vals_in,
                uint32_t* vals_out, size_t n_host, const uint32_t* d_n, size_t capacity, int begin_bit, int end_bit,
                cudaStream_t s);
int launch_ranges(lcgs_b200_ctx* ctx, const uint64_t* keys, size_t n_host, const uint32_t* d_n, size_t capacity,
                  uint32_t* ranges, int num_tiles, cudaStream_t s, bool cleared = false);
int launch_blend(lcgs_b200_ctx* ctx, int W, int H, const float* bg, const uint32_t* ranges, const uint32_t* point_list,
                 const float4* records, const uint32_t* d_num_rendered, float* img, uint8_t* rgb8, int row0, int row1,
                 cudaStream_t s, const float* depth = nullptr, float* out_alpha = nullptr, float* out_depth = nullptr,
                 uint32_t* out_n = nullptr);
int launch_transpose_rgba8(lcgs_b200_ctx* ctx, int W, int H, const float* img, uint8_t* rgba, cudaStream_t s);
int launch_scene_prepare(lcgs_b200_ctx* ctx, int P, const float* opacity, float* consts, cudaStream_t s);
int launch_tile_order(lcgs_b200_ctx* ctx, const uint32_t* ranges, int num_tiles, const uint32_t* d_num_rendered,
                      size_t list_capacity, cudaStream_t s);
// lcgs_b200_render_backward of a whole frame (backward.cu); arguments checked by the caller
int launch_render_backward(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                           const lcgs_b200_frame* fr, const lcgs_b200_grad* gr, cudaStream_t s);
int launch_peer_signal(lcgs_b200_ctx* ctx, uint32_t* flag, uint32_t value, cudaStream_t s);
int launch_peer_wait(lcgs_b200_ctx* ctx, const uint32_t* flag, uint32_t value, uint32_t timeout_ms, cudaStream_t s);
int launch_checksum_u32(lcgs_b200_ctx* ctx, const void* data, size_t num_words, uint64_t* out, cudaStream_t s);
int launch_fill_u32(lcgs_b200_ctx* ctx, uint32_t* buf, size_t n, uint32_t v, cudaStream_t s);
int launch_fill_u64(lcgs_b200_ctx* ctx, uint64_t* buf, size_t n, uint64_t v, cudaStream_t s);
int launch_fill_f32(lcgs_b200_ctx* ctx, float* buf, size_t n, float v, cudaStream_t s);

}  // namespace lcgs_b200
