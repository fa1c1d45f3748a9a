// capi.cu -- the extern "C" boundary (include/lcgs_b200.h): context, host-side camera helpers,
// per-stage entry points and the two whole-frame orchestrations.
#include <math.h>
#include <new>
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

using namespace lcgs_b200;

namespace lcgs_b200 {

int ws_reserve(lcgs_b200_ctx* ctx, Workspace& ws, size_t bytes)
{
    if (bytes <= ws.bytes) return LCGS_B200_OK;
    // grow geometrically, never shrink (lcgs/src/gs_tile_splatter/impl.cpp:37-44)
    size_t want = ws.bytes * 2 > bytes ? ws.bytes * 2 : bytes;
    if (ws.ptr) {
        LCGS_CUDA_CHECK(ctx, cudaDeviceSynchronize());
        LCGS_CUDA_CHECK(ctx, cudaFree(ws.ptr));
        ws.ptr   = nullptr;
        ws.bytes = 0;
    }
    cudaError_t e = cudaMalloc(&ws.ptr, want);
    if (e != cudaSuccess && want > bytes) {
        (void)cudaGetLastError();
        want = bytes;
        e    = cudaMalloc(&ws.ptr, want);
    }
    LCGS_CUDA_CHECK(ctx, e);
    ws.bytes = want;
    return LCGS_B200_OK;
}

static inline cudaStream_t as_stream(lcgs_b200_stream s) { return reinterpret_cast<cudaStream_t>(s); }

static int enter(lcgs_b200_ctx* ctx)
{
    if (!ctx) return LCGS_B200_ERR_INVALID;
    LCGS_CUDA_CHECK(ctx, cudaSetDevice(ctx->device));
    return LCGS_B200_OK;
}

static inline int ceil_log2(uint32_t v)
{
    int b = 0;
    while ((1ull << b) < (unsigned long long)v) b++;
    return b;
}

static inline bool aligned(const void* p, size_t a) { return (((uintptr_t)p) & (a - 1)) == 0; }

static void mark(lcgs_b200_ctx* ctx, cudaStream_t s)
{
    if (ctx->profiling && ctx->ev_count < 16) cudaEventRecord(ctx->ev[ctx->ev_count++], s);
}

struct FrameGeom {
    int      W, H;
    uint32_t gx, gy;
    int      row0, row1;
    int      num_tiles;
    int      end_bit;
};

static int frame_geom(lcgs_b200_ctx* ctx, const lcgs_b200_frame* fr, FrameGeom* g)
{
    LCGS_REQUIRE(ctx, fr && fr->width > 0 && fr->height > 0, "frame: bad resolution");
    g->W    = fr->width;
    g->H    = fr->height;
    g->gx   = (uint32_t)((fr->width + 15) / 16);
    g->gy   = (uint32_t)((fr->height + 15) / 16);
    g->row0 = fr->tile_row_begin;
    g->row1 = fr->tile_row_end < 0 ? (int)g->gy : fr->tile_row_end;
    LCGS_REQUIRE(ctx, g->row0 >= 0 && g->row1 <= (int)g->gy && g->row0 <= g->row1, "frame: bad tile row band");
    // the fused path packs tile rects into 16-bit fields (preprocess.cu) and tile ids into 32 bits
    LCGS_REQUIRE(ctx, g->gx < 65536u && g->gy < 65536u, "frame: more than 65535 tiles per row / column");
    g->num_tiles = (int)g->gx * (g->row1 - g->row0);
    // keys are (tile << 32) | depth bits: bits above 32 + ceil(log2(tiles)) are zero, so restricting
    // the sorted bit range is result-identical to the reference's 64-bit sort
    g->end_bit = 32 + ceil_log2((uint32_t)(g->num_tiles > 1 ? g->num_tiles : 1));
    return LCGS_B200_OK;
}

static int check_frame_lists(lcgs_b200_ctx* ctx, const lcgs_b200_frame* fr)
{
    LCGS_REQUIRE(ctx, fr->depth && fr->tiles_touched && fr->point_offsets && fr->radii, "frame: missing per-Gaussian buffer");
    LCGS_REQUIRE(ctx, fr->point_list_keys_unsorted && fr->point_list_unsorted && fr->point_list_keys && fr->point_list,
                 "frame: missing instance list");
    LCGS_REQUIRE(ctx, fr->ranges && fr->target_img, "frame: missing ranges / target_img");
    LCGS_REQUIRE(ctx, aligned(fr->point_list_keys_unsorted, 8) && aligned(fr->point_list_keys, 8) && aligned(fr->ranges, 8),
                 "frame: keys / ranges must be 8-byte aligned");
    LCGS_REQUIRE(ctx, aligned(fr->target_alpha, 4) && aligned(fr->target_depth, 4) && aligned(fr->target_n_contrib, 4),
                 "frame: target_alpha / target_depth / target_n_contrib must be 4-byte aligned");
    return LCGS_B200_OK;
}

// Layout of the fused path's order workspace (all arrays have P entries).
struct OrderWs {
    uint2*    rects;
    uint32_t *ckeys, *cvals, *skeys, *svals;
};
static OrderWs order_ws_views(lcgs_b200_ctx* ctx, int P)
{
    OrderWs o;
    char*   base = (char*)ctx->order_ws.ptr;
    const size_t n = (size_t)(P > 0 ? P : 1);
    o.rects    = (uint2*)base;
    o.ckeys    = (uint32_t*)(base + 8 * n);
    o.cvals    = o.ckeys + n;
    o.skeys    = o.cvals + n;
    o.svals    = o.skeys + n;
    return o;
}

static uint32_t big_threshold() { return (uint32_t)LCGS_TUNE_INT("LCGS_EMIT_BIG", (int)kBigThreshold); }

// The fused frame's plan (frame_plan.cuh): both sorts' geometry, then every scratch region, ticket and histogram placed in
// the workspaces reserve_all reserved, before the first kernel.
static int plan_frame(lcgs_b200_ctx* ctx, int P, const lcgs_b200_frame* fr, const FrameGeom& g, FramePlan* fp)
{
    int rc;
    if ((rc = sort_plan_geometry(ctx, (size_t)P, 0, 32, &fp->depth))) return rc;
    if ((rc = sort_plan_geometry(ctx, fr->list_capacity, 32, g.end_bit, &fp->tile))) return rc;
    const char* err = place_frame(fp, P, fr->list_capacity, big_threshold(), ctx->scan_ws, ctx->sort_ws, ctx->emit_ws,
                                  ctx->d_scalars, fr->ranges, (size_t)g.num_tiles);
    LCGS_REQUIRE(ctx, !err, err);
    return LCGS_B200_OK;
}

// scan -> [depth sort of the Gaussians] -> duplicate -> sort -> ranges -> blend, all on device-resident counts.
// depth_ordered = false: the reference's data flow (emit in index order, sort all key bits).
// depth_ordered = true : sort the Gaussians by depth, emit in that order, stable-sort by tile bits only;
//                        sorted keys / values / ranges are bit-identical (see scan.cu).
static int splat_tail(lcgs_b200_ctx* ctx, int P, const lcgs_b200_frame* fr, const FrameGeom& g, const float* means_pix,
                      bool depth_ordered, cudaStream_t s)
{
    int       rc;
    uint32_t* d_n = ctx->d_scalars + LCGS_SCALAR_NUM_RENDERED;
    uint32_t* d_m = ctx->d_scalars + LCGS_SCALAR_NUM_TOUCHING;
    if (depth_ordered) {
        const OrderWs o = order_ws_views(ctx, P);
        // Depth keys are stored relative to bits(0.2f) (kDepthKeyBase): 27 bits for any depth below 13107, so the
        // fourth 9-bit pass normally skips itself.  The compaction kernel also fills the depth sort's digit
        // histograms, the emission kernel those of the tile sort.
        FramePlan fp;
        if ((rc = plan_frame(ctx, P, fr, g, &fp))) return rc;
        if ((rc = launch_clear(ctx, fp.clear, s))) return rc;
        if ((rc = launch_scan_compact(ctx, fr->tiles_touched, fr->depth, P, fr->point_offsets, o.ckeys, o.cvals, d_n, d_m, fp, s)))
            return rc;
        mark(ctx, s);
        SortedPairsU32 sorted;
        if ((rc = sort_run_u32(ctx, fp.depth, o.ckeys, o.skeys, o.cvals, o.svals, d_m, (size_t)P, &sorted, s))) return rc;
        mark(ctx, s);
        if ((rc = launch_duplicate_keys_sorted(ctx, d_m, P, g.W, g.H, g.row1 - g.row0, sorted, o.rects, fr->point_list_keys_unsorted,
                                               fr->point_list_unsorted, fr->list_capacity, g.row0, fp, s)))
            return rc;
        mark(ctx, s);
        if ((rc = sort_run_u64(ctx, fp.tile, fr->point_list_keys_unsorted, fr->point_list_keys, fr->point_list_unsorted,
                               fr->point_list, d_n, fr->list_capacity, s)))
            return rc;
        mark(ctx, s);
    } else {
        if ((rc = launch_scan(ctx, fr->tiles_touched, fr->point_offsets, (size_t)P, d_n, s))) return rc;
        mark(ctx, s);
        mark(ctx, s);  // no depth sort in the reference's data flow
        if ((rc = launch_duplicate_keys(ctx, P, g.W, g.H, means_pix, fr->point_offsets, fr->radii, fr->depth,
                                        fr->point_list_keys_unsorted, fr->point_list_unsorted, fr->list_capacity, g.row0,
                                        g.row1, s)))
            return rc;
        mark(ctx, s);
        if ((rc = launch_sort(ctx, fr->point_list_keys_unsorted, fr->point_list_keys, fr->point_list_unsorted,
                              fr->point_list, 0, d_n, fr->list_capacity, 0, g.end_bit, s)))
            return rc;
        mark(ctx, s);
    }
    if ((rc = launch_ranges(ctx, fr->point_list_keys, 0, d_n, fr->list_capacity, fr->ranges, g.num_tiles, s, depth_ordered))) return rc;
    mark(ctx, s);
    // tile schedule (longest list first) + the frame's capacity check, made on the device against the count
    if ((rc = launch_tile_order(ctx, fr->ranges, g.num_tiles, d_n, fr->list_capacity, s))) return rc;
    if ((rc = launch_blend(ctx, g.W, g.H, fr->bg_color, fr->ranges, fr->point_list, (const float4*)ctx->record_ws.ptr, d_n,
                           fr->target_img, fr->target_rgb8, g.row0, g.row1, s, fr->depth, fr->target_alpha, fr->target_depth,
                           fr->target_n_contrib)))
        return rc;
    mark(ctx, s);
    // count, overflow flag and the capacity it was tested against travel back together (in stream order, so
    // pipelined frames with different capacities and graph replays report their own)
    LCGS_CUDA_CHECK(ctx, cudaMemcpyAsync(ctx->h_scalars, ctx->d_scalars, LCGS_NUM_SCALARS * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    ctx->ev_valid = ctx->profiling ? ctx->ev_count : 0;
    return LCGS_B200_OK;
}

#ifdef LCGS_TUNING
int tuning_env_int(const char* name, int fallback)
{
    const char* e = getenv(name);
    return e ? atoi(e) : fallback;
}
#endif

static int reserve_all(lcgs_b200_ctx* ctx, int P, size_t max_instances)
{
    int rc;
    if (P > 0) {
        const FrameWsBytes b = frame_ws_bytes(P, max_instances, big_threshold());
        if ((rc = ws_reserve(ctx, ctx->record_ws, (size_t)P * kRecordFloat4s * sizeof(float4)))) return rc;
        if ((rc = ws_reserve(ctx, ctx->scan_ws, b.scan))) return rc;
        if ((rc = ws_reserve(ctx, ctx->order_ws, (size_t)P * 24))) return rc;
        if ((rc = ws_reserve(ctx, ctx->emit_ws, b.emit))) return rc;
        if ((rc = ws_reserve(ctx, ctx->sort_ws, b.sort))) return rc;
    } else if (max_instances > 0) {
        if ((rc = ws_reserve(ctx, ctx->sort_ws, sort_temp_bytes(max_instances)))) return rc;
    }
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200

// =================================================================================================
extern "C" {

int lcgs_b200_version(void) { return LCGS_B200_VERSION; }

const char* lcgs_b200_status_string(int status)
{
    switch (status) {
        case LCGS_B200_OK: return "ok";
        case LCGS_B200_ERR_INVALID: return "invalid argument";
        case LCGS_B200_ERR_CUDA: return "CUDA error";
        case LCGS_B200_ERR_CAPACITY: return "num_rendered exceeds list capacity";
        case LCGS_B200_ERR_NO_DEVICE: return "no CUDA device (there is no CPU fallback)";
        case LCGS_B200_ERR_UNSUPPORTED: return "unsupported";
        default: return "unknown status";
    }
}

int lcgs_b200_ctx_create(int device, lcgs_b200_ctx** out)
{
    if (!out) return LCGS_B200_ERR_INVALID;
    *out      = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        (void)cudaGetLastError();
        return LCGS_B200_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= count) return LCGS_B200_ERR_INVALID;
    lcgs_b200_ctx* ctx = new (std::nothrow) lcgs_b200_ctx();
    if (!ctx) return LCGS_B200_ERR_INVALID;
    ctx->device        = device;
    ctx->last_error[0] = 0;
    if (cudaSetDevice(device) != cudaSuccess) { delete ctx; return LCGS_B200_ERR_CUDA; }
    int sms = 0;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) == cudaSuccess && sms > 0) ctx->num_sms = sms;
    if (cudaMalloc(&ctx->d_scalars, LCGS_NUM_SCALARS * sizeof(uint32_t)) != cudaSuccess ||
        cudaMemset(ctx->d_scalars, 0, LCGS_NUM_SCALARS * sizeof(uint32_t)) != cudaSuccess ||
        cudaMallocHost(&ctx->h_scalars, LCGS_NUM_SCALARS * sizeof(uint32_t)) != cudaSuccess) {
        lcgs_b200_ctx_destroy(ctx);
        return LCGS_B200_ERR_CUDA;
    }
    memset(ctx->h_scalars, 0, LCGS_NUM_SCALARS * sizeof(uint32_t));
    for (int i = 0; i < 16; i++) ctx->ev[i] = nullptr;
    *out = ctx;
    return LCGS_B200_OK;
}

int lcgs_b200_ctx_destroy(lcgs_b200_ctx* ctx)
{
    if (!ctx) return LCGS_B200_OK;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (ctx->d_scalars) cudaFree(ctx->d_scalars);
    if (ctx->h_scalars) cudaFreeHost(ctx->h_scalars);
    if (ctx->scan_ws.ptr) cudaFree(ctx->scan_ws.ptr);
    if (ctx->sort_ws.ptr) cudaFree(ctx->sort_ws.ptr);
    if (ctx->record_ws.ptr) cudaFree(ctx->record_ws.ptr);
    if (ctx->order_ws.ptr) cudaFree(ctx->order_ws.ptr);
    if (ctx->tile_order_ws.ptr) cudaFree(ctx->tile_order_ws.ptr);
    if (ctx->emit_ws.ptr) cudaFree(ctx->emit_ws.ptr);
    if (ctx->grad_ws.ptr) cudaFree(ctx->grad_ws.ptr);
    if (ctx->pose_ws.ptr) cudaFree(ctx->pose_ws.ptr);
    if (ctx->ssim_ws.ptr) cudaFree(ctx->ssim_ws.ptr);
    for (int i = 0; i < 16; i++)
        if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (int i = 0; i < 3; i++)
        if (ctx->ev_sort[i]) cudaEventDestroy(ctx->ev_sort[i]);
    delete ctx;
    return LCGS_B200_OK;
}

int lcgs_b200_ctx_reserve(lcgs_b200_ctx* ctx, int num_gaussians, size_t max_instances)
{
    int rc = enter(ctx);
    if (rc) return rc;
    return reserve_all(ctx, num_gaussians, max_instances);
}

const char* lcgs_b200_last_error(const lcgs_b200_ctx* ctx) { return ctx ? ctx->last_error : "null context"; }

// ---- camera helpers (host) ------------------------------------------------------------------------

static inline float dot3(const float* a, const float* b) { return (a[0] * b[0] + a[1] * b[1]) + a[2] * b[2]; }
static inline void  cross3(const float* a, const float* b, float* o)
{
    const float x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
    o[0] = x; o[1] = y; o[2] = z;
}
static inline void normalize3(const float* v, float* o)
{
    const float inv = 1.0f / sqrtf(dot3(v, v));
    o[0] = v[0] * inv; o[1] = v[1] * inv; o[2] = v[2] * inv;
}

int lcgs_b200_get_lookat_cam(const float pos[3], const float target[3], const float world_up[3], lcgs_b200_camera* cam)
{
    if (!pos || !target || !world_up || !cam) return LCGS_B200_ERR_INVALID;
    const float d[3] = { target[0] - pos[0], target[1] - pos[1], target[2] - pos[2] };
    float       c[3];
    for (int i = 0; i < 3; i++) cam->position[i] = pos[i];
    normalize3(d, cam->front);
    cross3(cam->front, world_up, c);
    normalize3(c, cam->right);
    cross3(cam->right, cam->front, c);
    normalize3(c, cam->up);
    cam->fov = 60.0f; cam->aspect_ratio = 1.0f; cam->width = 512; cam->height = 512;
    return LCGS_B200_OK;
}

int lcgs_b200_local_to_world_matrix(const lcgs_b200_camera* cam, float m[16])
{
    if (!cam || !m) return LCGS_B200_ERR_INVALID;
    for (int r = 0; r < 3; r++) {
        m[0 + r] = cam->right[r]; m[4 + r] = cam->up[r]; m[8 + r] = cam->front[r]; m[12 + r] = cam->position[r];
    }
    m[3] = 0.f; m[7] = 0.f; m[11] = 0.f; m[15] = 1.f;
    return LCGS_B200_OK;
}

int lcgs_b200_world_to_local_matrix(const lcgs_b200_camera* cam, float m[16])
{
    if (!cam || !m) return LCGS_B200_ERR_INVALID;
    for (int c = 0; c < 3; c++) {
        m[c * 4 + 0] = cam->right[c]; m[c * 4 + 1] = cam->up[c]; m[c * 4 + 2] = cam->front[c]; m[c * 4 + 3] = 0.f;
    }
    m[12] = -dot3(cam->position, cam->right);
    m[13] = -dot3(cam->position, cam->up);
    m[14] = -dot3(cam->position, cam->front);
    m[15] = 1.f;
    return LCGS_B200_OK;
}

int lcgs_b200_projection_matrix(float tanfovx, float tanfovy, float znear, float zfar, float m[16])
{
    if (!m) return LCGS_B200_ERR_INVALID;
    const float zsign = 1.0f, z_range = zfar - znear;
    for (int i = 0; i < 16; i++) m[i] = 0.f;
    m[0]  = 1.0f / tanfovx;
    m[5]  = 1.0f / tanfovy;
    m[10] = zfar / z_range * zsign;
    m[11] = zsign;
    m[14] = -zfar * znear / z_range;
    return LCGS_B200_OK;
}

int lcgs_b200_view_params_from_camera(const lcgs_b200_camera* cam, lcgs_b200_view_params* vp)
{
    if (!cam || !vp) return LCGS_B200_ERR_INVALID;
    const float fovy    = cam->fov / 180.0f * 3.1415926536f;
    const float tanfovy = tanf(fovy * 0.5f);
    const float tanfovx = tanfovy * cam->aspect_ratio;
    lcgs_b200_world_to_local_matrix(cam, vp->view);
    lcgs_b200_projection_matrix(tanfovx, tanfovy, 0.1f, 100.0f, vp->proj);
    vp->tanfovx = tanfovx;
    vp->tanfovy = tanfovy;
    vp->focalx  = (float)cam->width / (2.0f * tanfovx);
    vp->focaly  = (float)cam->height / (2.0f * tanfovy);
    for (int i = 0; i < 3; i++) vp->cam_pos[i] = cam->position[i];
    vp->width  = cam->width;
    vp->height = cam->height;
    return LCGS_B200_OK;
}

// ---- stage entry points -----------------------------------------------------------------------------

int lcgs_b200_sh_process(lcgs_b200_ctx* ctx, int P, int sh_deg, const float cam_pos[3], const float* pos, const float* sh,
                         float* color, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && sh_deg >= -1 && sh_deg <= 3, "sh_process: bad P / degree");
    LCGS_REQUIRE(ctx, P == 0 || (cam_pos && pos && sh && color), "sh_process: null pointer");
    return launch_sh(ctx, P, sh_deg, cam_pos, pos, sh, color, as_stream(stream));
}

int lcgs_b200_project(lcgs_b200_ctx* ctx, int P, const float* pos, const float* scale, const float* rotq,
                      float scale_modifier, const lcgs_b200_view_params* vp, float* means_2d, float* depth,
                      float* covs_2d, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && vp, "project: bad arguments");
    LCGS_REQUIRE(ctx, P == 0 || (pos && scale && rotq && means_2d && depth && covs_2d), "project: null pointer");
    ViewParams v;
    memcpy(&v, vp, sizeof(v));
    return launch_project(ctx, P, pos, scale, rotq, scale_modifier, v, means_2d, depth, covs_2d, as_stream(stream));
}

int lcgs_b200_allocate_tiles(lcgs_b200_ctx* ctx, int P, int width, int height, const float* depth, float* means_2d,
                             float* covs_2d, uint32_t* tiles_touched, int32_t* radii, int row0, int row1,
                             lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && width > 0 && height > 0, "allocate_tiles: bad sizes");
    LCGS_REQUIRE(ctx, P == 0 || (depth && means_2d && covs_2d && tiles_touched && radii), "allocate_tiles: null pointer");
    return launch_allocate_tiles(ctx, P, width, height, depth, means_2d, covs_2d, tiles_touched, radii, row0, row1,
                                 as_stream(stream));
}

int lcgs_b200_fill_u32(lcgs_b200_ctx* ctx, uint32_t* buf, size_t n, uint32_t v, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, n == 0 || buf, "fill: null pointer");
    return launch_fill_u32(ctx, buf, n, v, as_stream(stream));
}
int lcgs_b200_fill_u64(lcgs_b200_ctx* ctx, uint64_t* buf, size_t n, uint64_t v, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, n == 0 || buf, "fill: null pointer");
    return launch_fill_u64(ctx, buf, n, v, as_stream(stream));
}
int lcgs_b200_fill_f32(lcgs_b200_ctx* ctx, float* buf, size_t n, float v, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, n == 0 || buf, "fill: null pointer");
    return launch_fill_f32(ctx, buf, n, v, as_stream(stream));
}

size_t lcgs_b200_scan_temp_bytes(size_t num_items)
{
    return ((num_items + kScanTile - 1) / kScanTile) * sizeof(unsigned long long);
}

int lcgs_b200_scan_inclusive_u32(lcgs_b200_ctx* ctx, const uint32_t* in, uint32_t* out, size_t n, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, n == 0 || (in && out), "scan: null pointer");
    return launch_scan(ctx, in, out, n, nullptr, as_stream(stream));
}

int lcgs_b200_duplicate_keys(lcgs_b200_ctx* ctx, int P, int width, int height, const float* means_2d_pix,
                             const uint32_t* point_offsets, const int32_t* radii, const float* depth, uint64_t* keys,
                             uint32_t* vals, size_t capacity, int row0, int row1, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && width > 0 && height > 0, "duplicate_keys: bad sizes");
    LCGS_REQUIRE(ctx, P == 0 || (means_2d_pix && point_offsets && radii && depth), "duplicate_keys: null pointer");
    LCGS_REQUIRE(ctx, capacity == 0 || (keys && vals), "duplicate_keys: null list");
    LCGS_REQUIRE(ctx, aligned(means_2d_pix, 8) && aligned(keys, 8), "duplicate_keys: means_2d / keys must be 8-byte aligned");
    return launch_duplicate_keys(ctx, P, width, height, means_2d_pix, point_offsets, radii, depth, keys, vals, capacity,
                                 row0, row1, as_stream(stream));
}

size_t lcgs_b200_sort_temp_bytes(size_t num_items) { return sort_temp_bytes(num_items); }

int lcgs_b200_sort_pairs_u64_u32(lcgs_b200_ctx* ctx, const uint64_t* keys_in, uint64_t* keys_out, const uint32_t* vals_in,
                                 uint32_t* vals_out, size_t n, int begin_bit, int end_bit, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, n == 0 || (keys_in && keys_out && vals_in && vals_out), "sort: null pointer");
    LCGS_REQUIRE(ctx, aligned(keys_in, 8) && aligned(keys_out, 8), "sort: keys must be 8-byte aligned");
    return launch_sort(ctx, keys_in, keys_out, vals_in, vals_out, n, nullptr, n, begin_bit, end_bit, as_stream(stream));
}

int lcgs_b200_tile_ranges(lcgs_b200_ctx* ctx, const uint64_t* keys_sorted, size_t n, uint32_t* ranges, int num_tiles,
                          lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, num_tiles >= 0 && (num_tiles == 0 || ranges) && (n == 0 || keys_sorted), "tile_ranges: bad arguments");
    return launch_ranges(ctx, keys_sorted, n, nullptr, n, ranges, num_tiles, as_stream(stream));
}

int lcgs_b200_blend(lcgs_b200_ctx* ctx, int P, int width, int height, const float bg_color[3], const uint32_t* ranges,
                    const uint32_t* point_list, const float* means_2d, const float* conic, const float* opacity,
                    const float* color, const uint32_t* tiles_touched, float* target_img, int row0, int row1,
                    lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && width > 0 && height > 0 && bg_color && ranges && target_img, "blend: bad arguments");
    LCGS_REQUIRE(ctx, P == 0 || (point_list && means_2d && conic && opacity && color), "blend: null pointer");
    LCGS_REQUIRE(ctx, aligned(ranges, 8), "blend: ranges must be 8-byte aligned");
    if ((rc = ws_reserve(ctx, ctx->record_ws, (size_t)(P > 0 ? P : 1) * kRecordFloat4s * sizeof(float4)))) return rc;
    cudaStream_t s = as_stream(stream);
    if ((rc = launch_build_records(ctx, P, means_2d, conic, opacity, nullptr, color, tiles_touched,
                                   (float4*)ctx->record_ws.ptr, s)))
        return rc;
    const int gx = (width + 15) / 16, gy = (height + 15) / 16;
    if ((rc = launch_tile_order(ctx, ranges, gx * ((row1 < 0 ? gy : row1) - row0), nullptr, 0, s))) return rc;
    return launch_blend(ctx, width, height, bg_color, ranges, point_list, (const float4*)ctx->record_ws.ptr, nullptr,
                        target_img, nullptr, row0, row1, s);
}

// ---- whole frame ----------------------------------------------------------------------------------------

int lcgs_b200_splat_forward(lcgs_b200_ctx* ctx, int P, const float* opacity, const lcgs_b200_frame* fr,
                            lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    FrameGeom g;
    if ((rc = frame_geom(ctx, fr, &g))) return rc;
    if ((rc = check_frame_lists(ctx, fr))) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && (P == 0 || (opacity && fr->means_2d && fr->conic && fr->color)),
                 "splat_forward: means_2d / conic / color / opacity are required");
    LCGS_REQUIRE(ctx, aligned(fr->means_2d, 8), "splat_forward: means_2d must be 8-byte aligned");
    if ((rc = reserve_all(ctx, P > 0 ? P : 1, fr->list_capacity))) return rc;
    cudaStream_t s = as_stream(stream);
    ctx->ev_count  = 0;
    mark(ctx, s);
    if ((rc = launch_allocate_tiles(ctx, P, g.W, g.H, fr->depth, fr->means_2d, fr->conic, fr->tiles_touched, fr->radii,
                                    g.row0, g.row1, s)))
        return rc;
    if ((rc = launch_build_records(ctx, P, fr->means_2d, fr->conic, opacity, nullptr, fr->color, fr->tiles_touched,
                                   (float4*)ctx->record_ws.ptr, s)))
        return rc;
    mark(ctx, s);
    return splat_tail(ctx, P, fr, g, fr->means_2d, false, s);
}

int lcgs_b200_render(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                     const lcgs_b200_frame* fr, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, sc && vp && fr, "render: null argument");
    FrameGeom g;
    if ((rc = frame_geom(ctx, fr, &g))) return rc;
    if ((rc = check_frame_lists(ctx, fr))) return rc;
    const int P = sc->num_gaussians;
    LCGS_REQUIRE(ctx, P >= 0 && sc->sh_deg >= 0 && sc->sh_deg <= 3, "render: bad scene");
    LCGS_REQUIRE(ctx, P == 0 || (sc->pos && sc->scale && sc->rotq && sc->sh && sc->opacity), "render: null scene array");
    LCGS_REQUIRE(ctx, aligned(sc->rotq, 16) && aligned(sc->sh, 16), "render: rotq and sh must be 16-byte aligned");
    LCGS_REQUIRE(ctx, aligned(sc->alpha_consts, 8), "render: alpha_consts must be 8-byte aligned");
    LCGS_REQUIRE(ctx, aligned(fr->means_2d, 8), "render: means_2d must be 8-byte aligned");
    LCGS_REQUIRE(ctx, vp->width == fr->width && vp->height == fr->height, "render: view/frame resolution mismatch");
    if ((rc = reserve_all(ctx, P > 0 ? P : 1, fr->list_capacity))) return rc;
    cudaStream_t s = as_stream(stream);
    ctx->ev_count  = 0;
    mark(ctx, s);
    if ((rc = launch_preprocess_fused(ctx, sc, vp, fr, (float4*)ctx->record_ws.ptr, order_ws_views(ctx, P).rects, s))) return rc;
    mark(ctx, s);
    return splat_tail(ctx, P, fr, g, fr->means_2d, true, s);
}

int lcgs_b200_render_backward(lcgs_b200_ctx* ctx, const lcgs_b200_scene* sc, const lcgs_b200_view_params* vp,
                              const lcgs_b200_frame* fr, const lcgs_b200_grad* gr, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, sc && vp && fr && gr, "render_backward: null argument");
    FrameGeom g;
    if ((rc = frame_geom(ctx, fr, &g))) return rc;
    if (g.row0 != 0 || g.row1 != (int)g.gy) {
        snprintf(ctx->last_error, sizeof(ctx->last_error), "render_backward: tile-row bands are not supported");
        return LCGS_B200_ERR_UNSUPPORTED;
    }
    const int P = sc->num_gaussians;
    LCGS_REQUIRE(ctx, P >= 0 && sc->sh_deg >= 0 && sc->sh_deg <= 3, "render_backward: bad scene");
    LCGS_REQUIRE(ctx, vp->width == fr->width && vp->height == fr->height, "render_backward: view/frame resolution mismatch");
    LCGS_REQUIRE(ctx, fr->ranges && fr->target_img && gr->dl_dimg, "render_backward: missing ranges / target_img / dl_dimg");
    LCGS_REQUIRE(ctx, P == 0 || (sc->pos && sc->scale && sc->rotq && sc->sh && sc->opacity), "render_backward: null scene array");
    LCGS_REQUIRE(ctx, P == 0 || (fr->point_list && fr->means_2d && fr->conic && fr->color && fr->tiles_touched),
                 "render_backward: point_list / means_2d / conic / color / tiles_touched are required");
    LCGS_REQUIRE(ctx, aligned(sc->rotq, 16) && aligned(sc->sh, 16) && aligned(sc->alpha_consts, 8),
                 "render_backward: rotq and sh must be 16-byte, alpha_consts 8-byte aligned");
    LCGS_REQUIRE(ctx, aligned(fr->ranges, 8) && aligned(fr->means_2d, 8), "render_backward: ranges / means_2d must be 8-byte aligned");
    LCGS_REQUIRE(ctx, aligned(sc->pos, 4) && aligned(sc->scale, 4) && aligned(sc->opacity, 4) && aligned(fr->conic, 4) &&
                          aligned(fr->color, 4) && aligned(fr->tiles_touched, 4) && aligned(fr->point_list, 4) &&
                          aligned(fr->target_img, 4) && aligned(gr->dl_dimg, 4),
                 "render_backward: float / index buffers must be 4-byte aligned");
    LCGS_REQUIRE(ctx, aligned(gr->grad_pos, 4) && aligned(gr->grad_scale, 4) && aligned(gr->grad_rotq, 4) && aligned(gr->grad_sh, 4) &&
                          aligned(gr->grad_opacity, 4) && aligned(gr->grad_means_2d, 4) && aligned(gr->grad_conic, 4) &&
                          aligned(gr->grad_color, 4),
                 "render_backward: gradient buffers must be 4-byte aligned");
    LCGS_REQUIRE(ctx, !gr->dl_dalpha || fr->target_alpha, "render_backward: dl_dalpha needs the frame's target_alpha");
    LCGS_REQUIRE(ctx, !gr->dl_ddepth || (fr->target_depth && fr->depth),
                 "render_backward: dl_ddepth needs the frame's target_depth and depth");
    LCGS_REQUIRE(ctx, aligned(gr->dl_dalpha, 4) && aligned(gr->dl_ddepth, 4) && aligned(gr->grad_depth, 4) &&
                          (!gr->dl_dalpha || aligned(fr->target_alpha, 4)) &&
                          (!gr->dl_ddepth || (aligned(fr->target_depth, 4) && aligned(fr->depth, 4))),
                 "render_backward: aux plane buffers must be 4-byte aligned");
    LCGS_REQUIRE(ctx, aligned(gr->grad_view, 4) && aligned(gr->grad_cam_pos, 4),
                 "render_backward: grad_view / grad_cam_pos must be 4-byte aligned");
    return launch_render_backward(ctx, sc, vp, fr, gr, as_stream(stream));
}

int lcgs_b200_ssim(lcgs_b200_ctx* ctx, int width, int height, const float* img, const float* ref, float* ssim,
                   float* dssim_dimg, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, img && ref && ssim, "ssim: null img / ref / ssim");
    LCGS_REQUIRE(ctx, width > 0 && height > 0, "ssim: width and height must be positive");
    LCGS_REQUIRE(ctx, ((size_t)width + 31) / 32 * (((size_t)height + 31) / 32) <= 0x7fffffffu / 3,
                 "ssim: image too large");
    LCGS_REQUIRE(ctx, aligned(img, 4) && aligned(ref, 4) && aligned(ssim, 4) && aligned(dssim_dimg, 4),
                 "ssim: buffers must be 4-byte aligned");
    return launch_ssim(ctx, width, height, img, ref, ssim, dssim_dimg, as_stream(stream));
}

int lcgs_b200_num_rendered(lcgs_b200_ctx* ctx, lcgs_b200_stream stream, int* num_rendered)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, num_rendered, "num_rendered: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaStreamSynchronize(as_stream(stream)));
    const uint32_t n = ctx->h_scalars[LCGS_SCALAR_NUM_RENDERED];
    *num_rendered    = (int)n;  // the reference stores the uint count in an int (gs_tile_splatter.h:23)
    if (ctx->h_scalars[LCGS_SCALAR_OVERFLOW]) {  // set on the device by the frame itself
        snprintf(ctx->last_error, sizeof(ctx->last_error), "num_rendered %u exceeds list_capacity %u", n,
                 ctx->h_scalars[LCGS_SCALAR_CAPACITY]);
        return LCGS_B200_ERR_CAPACITY;
    }
    return LCGS_B200_OK;
}

int lcgs_b200_read_num_rendered_async(lcgs_b200_ctx* ctx, uint32_t* host_count, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, host_count, "read_num_rendered_async: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaMemcpyAsync(host_count, ctx->d_scalars + LCGS_SCALAR_NUM_RENDERED, sizeof(uint32_t),
                                         cudaMemcpyDeviceToHost, as_stream(stream)));
    return LCGS_B200_OK;
}

int lcgs_b200_read_image(lcgs_b200_ctx* ctx, const lcgs_b200_frame* fr, float* host_img, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, fr && host_img && fr->target_img, "read_image: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaMemcpyAsync(host_img, fr->target_img, (size_t)3 * fr->width * fr->height * sizeof(float),
                                         cudaMemcpyDeviceToHost, as_stream(stream)));
    return LCGS_B200_OK;
}

int lcgs_b200_read_image_rgb8(lcgs_b200_ctx* ctx, const lcgs_b200_frame* fr, uint8_t* host_rgb, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, fr && host_rgb && fr->target_rgb8, "read_image_rgb8: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaMemcpyAsync(host_rgb, fr->target_rgb8, (size_t)3 * fr->width * fr->height, cudaMemcpyDeviceToHost,
                                         as_stream(stream)));
    return LCGS_B200_OK;
}

int lcgs_b200_scene_prepare(lcgs_b200_ctx* ctx, int P, const float* opacity, float* consts, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, P >= 0 && (P == 0 || (opacity && consts)), "scene_prepare: bad arguments");
    LCGS_REQUIRE(ctx, aligned(consts, 8), "scene_prepare: consts must be 8-byte aligned");
    return launch_scene_prepare(ctx, P, opacity, consts, as_stream(stream));
}

int lcgs_b200_transpose_rgba8(lcgs_b200_ctx* ctx, int width, int height, const float* img_chw, uint8_t* rgba,
                              lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, width > 0 && height > 0 && img_chw && rgba, "transpose_rgba8: bad arguments");
    LCGS_REQUIRE(ctx, aligned(rgba, 4), "transpose_rgba8: rgba must be 4-byte aligned");
    return launch_transpose_rgba8(ctx, width, height, img_chw, rgba, as_stream(stream));
}

// ---- multi-GPU: peer-writable output buffers (CUDA IPC) ---------------------------------------------
static_assert(sizeof(cudaIpcMemHandle_t) == LCGS_B200_PEER_HANDLE_BYTES, "IPC handle size");

int lcgs_b200_peer_alloc(lcgs_b200_ctx* ctx, size_t bytes, void** dev_ptr, unsigned char handle[LCGS_B200_PEER_HANDLE_BYTES])
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, dev_ptr && handle && bytes > 0, "peer_alloc: bad argument");
    void* p = nullptr;
    LCGS_CUDA_CHECK(ctx, cudaMalloc(&p, bytes));
    cudaIpcMemHandle_t h;
    if (cudaMemset(p, 0, bytes) != cudaSuccess || cudaIpcGetMemHandle(&h, p) != cudaSuccess) {
        snprintf(ctx->last_error, sizeof(ctx->last_error), "peer_alloc: %s", cudaGetErrorString(cudaGetLastError()));
        cudaFree(p);
        return LCGS_B200_ERR_CUDA;
    }
    memcpy(handle, &h, sizeof(h));
    *dev_ptr = p;
    return LCGS_B200_OK;
}

int lcgs_b200_peer_open(lcgs_b200_ctx* ctx, const unsigned char handle[LCGS_B200_PEER_HANDLE_BYTES], void** dev_ptr)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, dev_ptr && handle, "peer_open: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    LCGS_CUDA_CHECK(ctx, cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return LCGS_B200_OK;
}

int lcgs_b200_peer_read(lcgs_b200_ctx* ctx, const void* dev_ptr, void* host_ptr, size_t bytes)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, dev_ptr && host_ptr, "peer_read: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaMemcpy(host_ptr, dev_ptr, bytes, cudaMemcpyDeviceToHost));
    return LCGS_B200_OK;
}

int lcgs_b200_peer_read_async(lcgs_b200_ctx* ctx, const void* dev_ptr, void* host_ptr, size_t bytes, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, dev_ptr && host_ptr, "peer_read_async: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaMemcpyAsync(host_ptr, dev_ptr, bytes, cudaMemcpyDeviceToHost, as_stream(stream)));
    return LCGS_B200_OK;
}

int lcgs_b200_peer_close(lcgs_b200_ctx* ctx, void* dev_ptr)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_CUDA_CHECK(ctx, cudaIpcCloseMemHandle(dev_ptr));
    return LCGS_B200_OK;
}

int lcgs_b200_peer_free(lcgs_b200_ctx* ctx, void* dev_ptr)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_CUDA_CHECK(ctx, cudaFree(dev_ptr));
    return LCGS_B200_OK;
}

int lcgs_b200_peer_signal(lcgs_b200_ctx* ctx, uint32_t* flag, uint32_t value, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, flag && aligned(flag, 4), "peer_signal: bad flag pointer");
    return launch_peer_signal(ctx, flag, value, as_stream(stream));
}

int lcgs_b200_peer_wait(lcgs_b200_ctx* ctx, const uint32_t* flag, uint32_t value, uint32_t timeout_ms, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, flag && aligned(flag, 4), "peer_wait: bad flag pointer");
    return launch_peer_wait(ctx, flag, value, timeout_ms, as_stream(stream));
}

int lcgs_b200_peer_error(lcgs_b200_ctx* ctx, uint32_t* timed_out)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, timed_out, "peer_error: null pointer");
    LCGS_CUDA_CHECK(ctx, cudaDeviceSynchronize());
    LCGS_CUDA_CHECK(ctx, cudaMemcpy(timed_out, ctx->d_scalars + LCGS_SCALAR_PEER_TIMEOUTS, sizeof(uint32_t), cudaMemcpyDeviceToHost));
    return LCGS_B200_OK;
}

int lcgs_b200_checksum_u32(lcgs_b200_ctx* ctx, const void* data, size_t num_words, uint64_t* out, lcgs_b200_stream stream)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, out && aligned(out, 8) && (num_words == 0 || (data && aligned(data, 16))), "checksum: bad arguments");
    return launch_checksum_u32(ctx, data, num_words, out, as_stream(stream));
}

int lcgs_b200_set_profiling(lcgs_b200_ctx* ctx, int enabled)
{
    int rc = enter(ctx);
    if (rc) return rc;
    if (enabled)
        for (int i = 0; i < 16; i++)
            if (!ctx->ev[i]) LCGS_CUDA_CHECK(ctx, cudaEventCreate(&ctx->ev[i]));
    if (enabled)
        for (int i = 0; i < 3; i++)
            if (!ctx->ev_sort[i]) LCGS_CUDA_CHECK(ctx, cudaEventCreate(&ctx->ev_sort[i]));
    ctx->profiling     = enabled ? 1 : 0;
    ctx->ev_valid      = 0;
    ctx->ev_sort_valid = 0;
    return LCGS_B200_OK;
}

int lcgs_b200_sort_breakdown(lcgs_b200_ctx* ctx, float* histogram_ms, float* passes_ms, int* num_passes)
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, histogram_ms && passes_ms && num_passes, "sort_breakdown: null pointer");
    LCGS_REQUIRE(ctx, ctx->ev_sort_valid, "sort_breakdown: no profiled sort (enable profiling first)");
    LCGS_CUDA_CHECK(ctx, cudaEventSynchronize(ctx->ev_sort[2]));
    LCGS_CUDA_CHECK(ctx, cudaEventElapsedTime(histogram_ms, ctx->ev_sort[0], ctx->ev_sort[1]));
    LCGS_CUDA_CHECK(ctx, cudaEventElapsedTime(passes_ms, ctx->ev_sort[1], ctx->ev_sort[2]));
    *num_passes = ctx->sort_passes;
    return LCGS_B200_OK;
}

int lcgs_b200_stage_times(lcgs_b200_ctx* ctx, float ms[LCGS_B200_NUM_STAGES])
{
    int rc = enter(ctx);
    if (rc) return rc;
    LCGS_REQUIRE(ctx, ms, "stage_times: null pointer");
    LCGS_REQUIRE(ctx, ctx->ev_valid == LCGS_B200_NUM_STAGES + 1, "stage_times: no profiled frame (enable profiling first)");
    LCGS_CUDA_CHECK(ctx, cudaEventSynchronize(ctx->ev[LCGS_B200_NUM_STAGES]));
    for (int i = 0; i < LCGS_B200_NUM_STAGES; i++) LCGS_CUDA_CHECK(ctx, cudaEventElapsedTime(&ms[i], ctx->ev[i], ctx->ev[i + 1]));
    return LCGS_B200_OK;
}

}  // extern "C"
