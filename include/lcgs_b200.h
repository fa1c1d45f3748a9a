/*
 * lcgs_b200.h -- C ABI of the B200-native forward splat-render path.
 *
 * Drop-in boundary for the hot path of LuisaGroup/LuisaComputeGaussianSplatting
 * (app/main.cpp:266-308 -> SHProcessor::process -> GSProjector::forward ->
 * GSTileSplatter::forward).  Every entry point cites the reference interface it replaces
 * (paths relative to the reference repository).  Plain pointers and sizes only: device pointers
 * are raw CUDA device addresses, `stream` is a cudaStream_t passed as void* (NULL = legacy default
 * stream).  All functions return an lcgs_b200_status (0 = ok, negative = error), never throw and
 * never fall back to the CPU: without a CUDA device ctx_create fails.
 *
 * Unless stated otherwise a call only ENQUEUES work on `stream` (like the reference's
 * CommandList-based entry points); nothing synchronises except lcgs_b200_num_rendered,
 * lcgs_b200_stage_times and ctx create/destroy/reserve.
 *
 * Threading: a context belongs to one host thread / one GPU at a time (the reference's modules
 * are not thread-safe either: mutable lazily-filled members, buffer_filler.h:56).  Use one context
 * per GPU, and ONE in-flight stream per context: the device scalars (num_rendered, tickets), the
 * look-back status words and the sort / record / order workspaces are per-context singletons, so
 * frames enqueued on two streams of one context would corrupt each other.  Frames enqueued back
 * to back on the same stream pipeline safely (every frame carries its own capacity check on the
 * device, see lcgs_b200_num_rendered).
 */
#ifndef LCGS_B200_H
#define LCGS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_MSC_VER)
#define LCGS_B200_API __declspec(dllexport)
#else
#define LCGS_B200_API __attribute__((visibility("default")))
#endif

#define LCGS_B200_VERSION 200 /* 0.2.0 */

typedef enum lcgs_b200_status {
    LCGS_B200_OK              = 0,
    LCGS_B200_ERR_INVALID     = -1, /* bad argument (null / misaligned pointer, negative size ...) */
    LCGS_B200_ERR_CUDA        = -2, /* a CUDA runtime call failed; see lcgs_b200_last_error */
    LCGS_B200_ERR_CAPACITY    = -3, /* num_rendered exceeds list_capacity (reference: unchecked overrun,
                                       app/main.cpp:245, gs_tile_splatter/impl.cpp:112-115) */
    LCGS_B200_ERR_NO_DEVICE   = -4, /* no CUDA device: there is no CPU fallback */
    LCGS_B200_ERR_UNSUPPORTED = -5
} lcgs_b200_status;

typedef struct lcgs_b200_ctx lcgs_b200_ctx;
typedef void*                lcgs_b200_stream; /* cudaStream_t */

/* lcgs::Camera -- lcgs/include/lcgs/util/camera.h:15-25 */
typedef struct lcgs_b200_camera {
    float position[3];
    float front[3];
    float up[3];
    float right[3];
    float fov;          /* degrees, vertical (default 60) */
    float aspect_ratio; /* width / height */
    int   width;
    int   height;
} lcgs_b200_camera;

/* What GSProjector::forward derives from the camera on the host before every launch
 * (lcgs/src/gs_projector/impl.cpp:34-42) plus the camera position SHProcessor::process passes
 * (lcgs/src/sh_preprocessor.cpp:182).  Matrices are column-major like luisa::float4x4. */
typedef struct lcgs_b200_view_params {
    float view[16];
    float proj[16];
    float tanfovx, tanfovy;
    float focalx, focaly;
    float cam_pos[3];
    int   width, height;
} lcgs_b200_view_params;

/* The device-resident Gaussian set: the five arrays app/main.cpp:180-223 uploads
 * (GaussiansData, app/gaussians.h:15-36).  pos [P][3], scale [P][3], rotq [P][4] = (r,x,y,z),
 * sh [P][(deg+1)^2][3], opacity [P]; all float32, post-activation.  rotq and sh must be 16-byte
 * aligned. */
typedef struct lcgs_b200_scene {
    int          num_gaussians;
    int          sh_deg; /* 0..3; app uses 3 */
    const float* pos;
    const float* scale;
    const float* rotq;
    const float* sh;
    const float* opacity;
    float        scale_modifier; /* GSProjectorInputProxy::scale_modifier, gs_projector.h:21 */
    /* extension, optional (NULL = computed per frame): per-Gaussian constants of the alpha test,
     * [P][2] float32 = (power threshold, log2(opacity)), a pure function of `opacity` written once per
     * scene by lcgs_b200_scene_prepare.  8-byte aligned.  Must be refreshed whenever opacity changes. */
    const float* alpha_consts;
} lcgs_b200_scene;

/* Caller-owned buffers of one frame: the union of GSTileSplatterInputProxy, GSTileSplatterAccelProxy
 * and GSSplatForwardOutputProxy (lcgs/include/lcgs/proxy.h:44-73), i.e. the 12 buffers
 * app/main.cpp:232-254 allocates.  Pointers marked optional may be NULL in lcgs_b200_render. */
typedef struct lcgs_b200_frame {
    int   width, height;
    float bg_color[3];
    /* GSTileSplatterInputProxy */
    float* means_2d; /* [P][2] NDC after project, pixels after allocate_tiles (in-place, Q7); 8-byte aligned;
                        optional in lcgs_b200_render */
    float* depth;    /* [P] */
    float* conic;    /* [P][3] optional; cov2d after project, conic after allocate_tiles (in-place) */
    float* color;    /* [P][3] optional */
    /* GSTileSplatterAccelProxy */
    uint32_t* tiles_touched;            /* [P]; 16-byte aligned buffers take the vector path, others a scalar one */
    uint32_t* point_offsets;            /* [P] inclusive sum */
    uint64_t* point_list_keys_unsorted; /* [L] */
    uint32_t* point_list_unsorted;      /* [L] */
    uint64_t* point_list_keys;          /* [L] */
    uint32_t* point_list;               /* [L] */
    uint32_t* ranges;                   /* [tiles][2] */
    size_t    list_capacity;            /* L (app/main.cpp:245 hard-codes 20 000 000) */
    /* GSSplatForwardOutputProxy */
    float*   target_img; /* planar CHW float32 [3][H][W] */
    int32_t* radii;      /* [P] */
    /* extension: render only tile rows [tile_row_begin, tile_row_end) (multi-GPU tile-row split);
     * tile_row_end < 0 means all rows.  Tile ids in keys/ranges are relative to tile_row_begin. */
    int tile_row_begin, tile_row_end;
    /* extension, optional (NULL = off): the blend kernel ALSO writes the image the app saves
     * (app/main.cpp:322-337): interleaved HWC uint8 [H][W][3], vertically flipped (row i = image row
     * H-1-i), uint8(v * 255) with truncation.  4x fewer bytes to read back than target_img. */
    uint8_t* target_rgb8;
    /* extension, optional (NULL = off; each plane on its own): per-pixel outputs of the blend, [H][W] in the row order
     * of target_img (not flipped), 4-byte aligned.  For a pixel whose front-to-back walk blends Gaussians i = 1..n with
     * weights w_i = T_i * alpha_i and ends with transmittance T (the factor of the background):
     *   target_alpha     = 1 - T                       (accumulated opacity)
     *   target_depth     = sum of w_i * depth[i]       (view depth, in blend order, not normalised: the expected
     *                                                   depth is target_depth / target_alpha where alpha > 0)
     *   target_n_contrib = n                           (pairs blended; entries skipped by the alpha test and the
     *                                                   entry that saturates the pixel are not counted)
     * Pixels no Gaussian reaches get 0.  A band of tile rows writes its own rows of these full-frame planes.  On an
     * empty whole frame (num_rendered == 0) the image is left untouched, but the planes are written as zeros.
     * Honoured by lcgs_b200_render and lcgs_b200_splat_forward. */
    float*    target_alpha;
    float*    target_depth;
    uint32_t* target_n_contrib;
} lcgs_b200_frame;

/* ---- library / context ------------------------------------------------------------------- */

LCGS_B200_API int         lcgs_b200_version(void);
LCGS_B200_API const char* lcgs_b200_status_string(int status);
/* replaces Context::create_device + Device::create_stream set-up and the three module create()
 * calls (app/main.cpp:162-163,173,213,227; kernels are AOT-compiled for sm_100a, nothing is JITed) */
LCGS_B200_API int         lcgs_b200_ctx_create(int device, lcgs_b200_ctx** out);
LCGS_B200_API int         lcgs_b200_ctx_destroy(lcgs_b200_ctx* ctx);
/* Pre-size the context-owned temp storage (replaces GSTileSplatter::ensure_scan_temp_buffer /
 * ensure_radix_sort_temp_buffer, lcgs/src/gs_tile_splatter/impl.cpp:31-61).  Called implicitly by
 * the stage functions; call it explicitly before CUDA-graph capture.  May synchronise. */
LCGS_B200_API int         lcgs_b200_ctx_reserve(lcgs_b200_ctx* ctx, int num_gaussians, size_t max_instances);
LCGS_B200_API const char* lcgs_b200_last_error(const lcgs_b200_ctx* ctx);

/* ---- host-side camera helpers (lcgs/include/lcgs/util/camera.h) ------------------------- */

/* get_lookat_cam, camera.h:74-82 (fov/aspect/width/height keep the struct defaults 60/1/512/512) */
LCGS_B200_API int lcgs_b200_get_lookat_cam(const float pos[3], const float target[3], const float world_up[3],
                                           lcgs_b200_camera* out);
LCGS_B200_API int lcgs_b200_local_to_world_matrix(const lcgs_b200_camera* cam, float m[16]); /* camera.h:27-36 */
LCGS_B200_API int lcgs_b200_world_to_local_matrix(const lcgs_b200_camera* cam, float m[16]); /* camera.h:38-51 */
LCGS_B200_API int lcgs_b200_projection_matrix(float tanfovx, float tanfovy, float znear, float zfar,
                                              float m[16]); /* camera.h:54-72 */
/* host prologue of GSProjector::forward, lcgs/src/gs_projector/impl.cpp:34-42 */
LCGS_B200_API int lcgs_b200_view_params_from_camera(const lcgs_b200_camera* cam, lcgs_b200_view_params* out);

/* ---- stage entry points (device pointers) ------------------------------------------------ */

/* SHProcessor::process, lcgs/include/lcgs/sh_preprocessor.h:30-37 / src/sh_preprocessor.cpp:169-188
 * (kernel shad_sh_process :159-166).  color[P][3] = clamp(SH(deg) . basis(dir) + 0.5, 0, 1). */
LCGS_B200_API int lcgs_b200_sh_process(lcgs_b200_ctx* ctx, int num_gaussians, int sh_deg, const float cam_pos[3],
                                       const float* pos, const float* sh, float* color, lcgs_b200_stream stream);

/* GSProjector::forward(use_focal=true), lcgs/include/lcgs/gs_projector.h:35-43 /
 * src/gs_projector/impl.cpp:26-68 (kernel shad_project_gs_focal, shader.cpp:82-139).  Writes
 * depth[P], means_2d[P][2] (NDC), covs_2d[P][3].  Near-culled Gaussians (z < 0.2) get zeros
 * (defined behaviour replacing the reference's stale-buffer quirk, SURVEY.md 9.7-Q6). */
LCGS_B200_API int lcgs_b200_project(lcgs_b200_ctx* ctx, int num_gaussians, const float* pos, const float* scale,
                                    const float* rotq, float scale_modifier, const lcgs_b200_view_params* vp,
                                    float* means_2d, float* depth, float* covs_2d, lcgs_b200_stream stream);

/* shad_allocate_tiles, lcgs/src/gs_tile_splatter/shader.cpp:102-163 (launched impl.cpp:87-100):
 * radii, tiles_touched; overwrites covs_2d <- conic and means_2d <- pixel coordinates in place. */
LCGS_B200_API int lcgs_b200_allocate_tiles(lcgs_b200_ctx* ctx, int num_gaussians, int width, int height,
                                           const float* depth, float* means_2d, float* covs_2d,
                                           uint32_t* tiles_touched, int32_t* radii, int tile_row_begin,
                                           int tile_row_end, lcgs_b200_stream stream);

/* BufferFiller::fill<uint>/<ulong>/<float>, lcgs/include/lcgs/util/buffer_filler.h:40-70 */
LCGS_B200_API int lcgs_b200_fill_u32(lcgs_b200_ctx* ctx, uint32_t* buf, size_t n, uint32_t v, lcgs_b200_stream stream);
LCGS_B200_API int lcgs_b200_fill_u64(lcgs_b200_ctx* ctx, uint64_t* buf, size_t n, uint64_t v, lcgs_b200_stream stream);
LCGS_B200_API int lcgs_b200_fill_f32(lcgs_b200_ctx* ctx, float* buf, size_t n, float v, lcgs_b200_stream stream);

/* lcpp DeviceScan<>::GetTempStorageBytes<uint> / InclusiveSum (call sites
 * lcgs/src/gs_tile_splatter/impl.cpp:34,104).  Temp storage is context-owned; the size query is
 * informational.  Single-pass decoupled look-back. */
LCGS_B200_API size_t lcgs_b200_scan_temp_bytes(size_t num_items);
LCGS_B200_API int    lcgs_b200_scan_inclusive_u32(lcgs_b200_ctx* ctx, const uint32_t* in, uint32_t* out, size_t n,
                                                  lcgs_b200_stream stream);

/* shad_copy_with_keys, lcgs/src/gs_tile_splatter/shader.cpp:26-69 (launched impl.cpp:120-131):
 * key = (tile_id << 32) | bits(depth), value = Gaussian index, written at point_offsets[i-1].
 * Entries past `capacity` are dropped (the reference overruns). */
LCGS_B200_API int lcgs_b200_duplicate_keys(lcgs_b200_ctx* ctx, int num_gaussians, int width, int height,
                                           const float* means_2d_pix, const uint32_t* point_offsets,
                                           const int32_t* radii, const float* depth, uint64_t* keys, uint32_t* vals,
                                           size_t capacity, int tile_row_begin, int tile_row_end,
                                           lcgs_b200_stream stream);

/* lcpp DeviceRadixSort<>::GetSortPairsTempStorageBytes<ulong,uint> / SortPairs<ulong,uint> (call
 * sites lcgs/src/gs_tile_splatter/impl.cpp:50,135-143).  Ascending, stable, bits [begin_bit,end_bit)
 * of the key (0,64 = the reference's call).  Inputs are preserved.  Onesweep LSD radix sort. */
LCGS_B200_API size_t lcgs_b200_sort_temp_bytes(size_t num_items);
LCGS_B200_API int    lcgs_b200_sort_pairs_u64_u32(lcgs_b200_ctx* ctx, const uint64_t* keys_in, uint64_t* keys_out,
                                                  const uint32_t* vals_in, uint32_t* vals_out, size_t n, int begin_bit,
                                                  int end_bit, lcgs_b200_stream stream);

/* BufferFiller::fill(ranges, 0) + shad_get_ranges, lcgs/src/gs_tile_splatter/impl.cpp:147-156,
 * shader.cpp:71-100.  ranges[num_tiles][2] = [start,end) per tile, (0,0) for empty tiles. */
LCGS_B200_API int lcgs_b200_tile_ranges(lcgs_b200_ctx* ctx, const uint64_t* keys_sorted, size_t n, uint32_t* ranges,
                                        int num_tiles, lcgs_b200_stream stream);

/* m_forward_render_shader, lcgs/src/gs_tile_splatter/shader.cpp:171-288 (launched impl.cpp:159-174).
 * means_2d are pixel coordinates, conic the inverse covariance (i.e. after allocate_tiles). */
LCGS_B200_API int lcgs_b200_blend(lcgs_b200_ctx* ctx, int num_gaussians, int width, int height, const float bg_color[3],
                                  const uint32_t* ranges, const uint32_t* point_list, const float* means_2d,
                                  const float* conic, const float* opacity, const float* color,
                                  const uint32_t* tiles_touched, float* target_img, int tile_row_begin,
                                  int tile_row_end, lcgs_b200_stream stream);

/* ---- whole-frame entry points ------------------------------------------------------------ */

/* GSTileSplatter::forward, lcgs/include/lcgs/gs_tile_splatter.h:28-35 / src/gs_tile_splatter/impl.cpp:63-180:
 * allocate_tiles -> scan -> copy_with_keys -> sort -> ranges -> render, from projector/SH outputs
 * held in `frame` (means_2d = NDC, conic = cov2d, depth, color) and `opacity`.  Unlike the
 * reference it does not synchronise five times: everything is enqueued, and the instance count is
 * fetched afterwards with lcgs_b200_num_rendered. */
LCGS_B200_API int lcgs_b200_splat_forward(lcgs_b200_ctx* ctx, int num_gaussians, const float* opacity,
                                          const lcgs_b200_frame* frame, lcgs_b200_stream stream);

/* One frame of the app's loop (app/main.cpp:266-299): SHProcessor::process + GSProjector::forward
 * + GSTileSplatter::forward with the three per-Gaussian passes fused into one kernel.  Enqueue
 * only, no allocation after lcgs_b200_ctx_reserve: capturable in a CUDA graph.  In this fused path
 * color is written only for Gaussians with tiles_touched > 0 (no other output depends on the
 * rest), NULL optional buffers are skipped, and the unsorted lists are emitted in depth order
 * (the Gaussians are sorted by depth first so that the instances only need a stable sort by tile):
 * point_list_keys_unsorted / point_list_unsorted hold the same pairs as the reference's in a
 * different order, while point_list_keys, point_list and ranges are bit-identical. */
LCGS_B200_API int lcgs_b200_render(lcgs_b200_ctx* ctx, const lcgs_b200_scene* scene, const lcgs_b200_view_params* vp,
                                   const lcgs_b200_frame* frame, lcgs_b200_stream stream);

/* ---- backward (no reference counterpart: the reference renders only) ------------------------
 *
 * Gradients of a scalar loss L of one whole frame's planar image target_img [3][H][W], rendered by
 * lcgs_b200_render, with respect to the five scene arrays as the forward uses them (after activation; chaining to
 * pre-activation parameters is the caller's).  Semantics, restated from the forward as written:
 *   blend, per pixel, over the entries i = 1..n the forward blended, in list order: w_i = T_i alpha_i,
 *     T_{i+1} = T_i (1 - alpha_i), C = sum w_i c_i + T_{n+1} bg; with G = dL/dC
 *       dL/dc_i = w_i G,  dL/dalpha_i = T_i (c_i . G) - (R_i . G) / (1 - alpha_i),  R_i = C - sum_{j<=i} w_j c_j.
 *     C is read back from target_img, so the backward walks front to back like the forward, with the same culling,
 *     ex2-based alpha and T (1 - alpha) < 1e-4 stop.  Entries the alpha test rejects and the entry that would saturate
 *     the pixel get no gradient.
 *   alpha = min(0.99, o e^power): zero gradient where the cap is active, else dalpha/do = alpha / o and
 *     dalpha/dpower = alpha; power = -1/2 (A dx^2 + C dy^2) - B dx dy, dx = mean_x - x_p (no half-pixel offset).
 *   preprocess: the projection, EWA covariance (unnormalised quaternion, scale_modifier), the +0.3 low-pass and
 *     det + 1e-6 of the conic, and the SH colour are differentiated as written.  The tx/ty clamp to +-1.3 tanfov and
 *     the [0,1] colour clamp (per channel) pass gradient only where inactive; the view direction of SH degree >= 1
 *     reaches pos.  radius, the tile rect, depth order and tiles_touched are discrete: a Gaussian with
 *     tiles_touched == 0 gets exactly zero in every output.  An empty frame gives all-zero gradients.
 *   aux planes (optional): with dl_dalpha = dL/dA and/or dl_ddepth = dL/dD for the frame's target_alpha
 *     A = 1 - T_{n+1} and target_depth D = sum w_i z_i (z_i = depth[i], the view depth), each plane is one more channel
 *     of the blend with colour 1 (alpha) or z_i (depth) and a background of 0: c_i . G above becomes
 *     c_i . G + z_i dL/dD + dL/dA, C . G becomes C . G + D dL/dD + A dL/dA, and dL/dz_i = sum over pixels w_i dL/dD,
 *     which reaches pos through the view transform.  A and D are read back from the frame, like C.  n_contrib is
 *     discrete and has no gradient.
 *   camera pose (optional grad_view / grad_cam_pos): with V = vp->view (column-major, p_view[k] =
 *     sum_c V[c*4+k] p[c] + V[12+k]) and dv = dL/dp_view of each Gaussian with tiles_touched > 0 (the depth plane's
 *     dL/dz included), summed over those Gaussians:
 *       dL/dV[c*4+k] = sum dv[k] p[c] (c < 3),  dL/dV[12+k] = sum dv[k],
 *       plus, through the EWA Jacobian's rows T0 = J00 V_col0 + J02 V_col2 and T1 = J11 V_col1 + J12 V_col2 of each
 *       Gaussian, dL/dV[r*4+0] += J00 dL/dT0[r], dL/dV[r*4+1] += J11 dL/dT1[r], dL/dV[r*4+2] += J02 dL/dT0[r] +
 *       J12 dL/dT1[r].  V[3], V[7], V[11] and V[15] never enter the forward and get 0.
 *     dL/dcam_pos = -(sum of the SH view-direction terms of dL/dpos): zero at SH degree 0 and for Gaussians whose
 *     three colour channels are all clamped.  proj, tanfov and focal are held fixed.  The alpha and depth planes reach
 *     the pose like the image does (with dl_ddepth the pose gradient includes the depth loss).  An empty frame gives
 *     zeros.  The per-Gaussian terms are summed per CTA and then, in double and a fixed order, over the CTAs.  The
 *     scene gradients are the same with or without the pose outputs.
 * Gradients are summed with float atomics: the last bits vary from run to run. */
typedef struct lcgs_b200_grad {
    const float* dl_dimg; /* [3][H][W], layout of target_img */
    /* scene gradients, each optional (NULL = not wanted); overwritten, not accumulated; 4-byte aligned */
    float *grad_pos, *grad_scale, *grad_rotq, *grad_sh, *grad_opacity;
    /* optional: gradients of the blend's per-Gaussian inputs -- pixel-space mean [P][2] (also the
       densification statistic trainers accumulate), conic [P][3], post-clamp colour [P][3] */
    float *grad_means_2d, *grad_conic, *grad_color;
    /* optional gradients of the aux planes, [H][W] in the layout of target_alpha / target_depth, 4-byte aligned
       (NULL = the plane is not in the loss).  dl_dalpha needs frame->target_alpha, dl_ddepth needs frame->target_depth
       and frame->depth, all as rendered with the frame. */
    const float* dl_dalpha;
    const float* dl_ddepth;
    /* optional [P]: dL/d(view depth) of each Gaussian, the blend's part (like grad_means_2d); all zeros without
       dl_ddepth */
    float* grad_depth;
    /* optional, device memory, 4-byte aligned, overwritten: dL/d(vp->view) [16] (column-major like vp->view;
       entries 3, 7, 11, 15 are 0) and dL/d(vp->cam_pos) [3] (through the SH view direction only). */
    float* grad_view;
    float* grad_cam_pos;
} lcgs_b200_grad;

/* Backward of one whole frame.  `scene`, `vp` and `frame` are those the frame was rendered with; the call reads only
 * the frame's point_list, ranges, means_2d, conic, color, tiles_touched and target_img (all required), plus the scene
 * and the view -- not the context's workspace from the forward, so any number of frames, on this context or another,
 * may be rendered between a frame and its backward as long as that frame's buffers are intact.  Enqueue only (no
 * host synchronisation except workspace growth).  With dl_dalpha or dl_ddepth it also reads target_alpha /
 * target_depth and depth.  LCGS_B200_ERR_INVALID for a NULL required pointer (a plane gradient without its plane
 * included) or a misaligned pointer, LCGS_B200_ERR_UNSUPPORTED for a tile-row band (whole frames only). */
LCGS_B200_API int lcgs_b200_render_backward(lcgs_b200_ctx* ctx, const lcgs_b200_scene* scene,
                                            const lcgs_b200_view_params* vp, const lcgs_b200_frame* frame,
                                            const lcgs_b200_grad* grad, lcgs_b200_stream stream);

/* SSIM of a planar image against a reference, and optionally its gradient (no reference counterpart: the reference
 * renders only; semantics: the 3DGS training loss's ssim(), see DESIGN).  img, ref: [3][H][W] float32, the layout of
 * target_img.  ssim: device float [1], overwritten with the mean SSIM.  dssim_dimg: optional [3][H][W], overwritten
 * with d(mean SSIM)/d(img), ready to be scaled into lcgs_b200_grad::dl_dimg.  All 4-byte aligned.  Enqueue only,
 * except workspace growth on the first call at a larger size; bit-reproducible.
 *   Window: 11 taps, sigma 1.5, applied separably per channel with zero padding of 5 (pixels outside the image are 0
 *   in every moment); C1 = 0.01^2, C2 = 0.03^2; the mean over the 3 H W channel pixels.  The reference image is a
 *   constant: there is no gradient with respect to it.  LCGS_B200_ERR_INVALID (nothing written) for a NULL img, ref
 *   or ssim, a width or height <= 0, or a misaligned pointer. */
LCGS_B200_API int lcgs_b200_ssim(lcgs_b200_ctx* ctx, int width, int height, const float* img, const float* ref,
                                 float* ssim, float* dssim_dimg, lcgs_b200_stream stream);

/* The value GSTileSplatter::forward returns (impl.cpp:179): synchronises `stream` (the one the
 * last whole-frame call was enqueued on) and stores that frame's num_rendered.  Returns LCGS_B200_ERR_CAPACITY if it exceeded
 * list_capacity (the frame's image is then incomplete).  The comparison is made ON THE DEVICE by the
 * frame itself (an overflow flag travels back with the count), so it is right for pipelined frames with
 * different capacities and for CUDA-graph replays. */
LCGS_B200_API int lcgs_b200_num_rendered(lcgs_b200_ctx* ctx, lcgs_b200_stream stream, int* num_rendered);

/* Pipelined variant of the above: enqueue a copy of the last enqueued frame's num_rendered into
 * (pinned) host memory on `stream`, without synchronising.  No capacity check. */
LCGS_B200_API int lcgs_b200_read_num_rendered_async(lcgs_b200_ctx* ctx, uint32_t* host_count, lcgs_b200_stream stream);

/* The read-back of app/main.cpp:313-315: enqueue a copy of the planar image to (pinned) host
 * memory on `stream`. */
LCGS_B200_API int lcgs_b200_read_image(lcgs_b200_ctx* ctx, const lcgs_b200_frame* frame, float* host_img,
                                       lcgs_b200_stream stream);

/* The same read-back for the fused uint8 image (frame->target_rgb8, 3*W*H bytes). */
LCGS_B200_API int lcgs_b200_read_image_rgb8(lcgs_b200_ctx* ctx, const lcgs_b200_frame* frame, uint8_t* host_rgb,
                                            lcgs_b200_stream stream);

/* Per-scene constants of the alpha test (see lcgs_b200_scene::alpha_consts): consts[P][2] =
 * (smallest power that passes alpha >= 1/255 for this opacity, log2(opacity)).  Enqueue only. */
LCGS_B200_API int lcgs_b200_scene_prepare(lcgs_b200_ctx* ctx, int num_gaussians, const float* opacity, float* consts,
                                          lcgs_b200_stream stream);

/* Display::_transpose_shader, app/display.cpp:30-39: planar CHW float image -> [H][W] RGBA8 (the BYTE4
 * framebuffer the viewer presents): unorm8 = round-to-nearest(clamp(v, 0, 1) * 255), alpha = 255, no flip. */
LCGS_B200_API int lcgs_b200_transpose_rgba8(lcgs_b200_ctx* ctx, int width, int height, const float* img_chw,
                                            uint8_t* rgba, lcgs_b200_stream stream);

/* ---- per-stage timing (the reference has a single wall clock, app/main.cpp:225-226,317) ---- */

#define LCGS_B200_NUM_STAGES 7 /* preprocess, scan, depth_sort, duplicate_keys, sort, ranges, blend */
LCGS_B200_API int lcgs_b200_set_profiling(lcgs_b200_ctx* ctx, int enabled);
/* Synchronises; ms[i] = device time of stage i of the last whole-frame call. */
LCGS_B200_API int lcgs_b200_stage_times(lcgs_b200_ctx* ctx, float ms[LCGS_B200_NUM_STAGES]);
/* Synchronises; device time of the last profiled sort split into its histogram kernel and its
 * `num_passes` onesweep launches (passes_ms / num_passes = average launch duration). */
LCGS_B200_API int lcgs_b200_sort_breakdown(lcgs_b200_ctx* ctx, float* histogram_ms, float* passes_ms, int* num_passes);

/* ---- multi-GPU: peer-writable output buffers (no reference counterpart: the reference drives one device,
 * app/main.cpp:162-163) ----
 *
 * One process per GPU.  The rank that assembles the result owns a device buffer every other rank can
 * WRITE with plain stores over NVLink (CUDA IPC + peer access): a rank passes the opened pointer (plus the
 * byte offset of its slot) as `target_img`, and the blend kernel's image stores are the transfer -- the
 * gather of finished frames / tile-row strips needs no separate collective or staging copy.  The owner
 * may read a slot after the writer's stream has finished its frame and the ranks have met at a barrier. */
#define LCGS_B200_PEER_HANDLE_BYTES 64
/* Owner: allocate `bytes` of zeroed device memory and export its interprocess handle. */
LCGS_B200_API int lcgs_b200_peer_alloc(lcgs_b200_ctx* ctx, size_t bytes, void** dev_ptr,
                                       unsigned char handle[LCGS_B200_PEER_HANDLE_BYTES]);
/* Other ranks (other processes, other GPUs of the node): map the owner's buffer; enables peer access. */
LCGS_B200_API int lcgs_b200_peer_open(lcgs_b200_ctx* ctx, const unsigned char handle[LCGS_B200_PEER_HANDLE_BYTES],
                                      void** dev_ptr);
/* Owner: synchronous copy of `bytes` from the buffer (dev_ptr may point anywhere inside it) to host memory. */
LCGS_B200_API int lcgs_b200_peer_read(lcgs_b200_ctx* ctx, const void* dev_ptr, void* host_ptr, size_t bytes);
/* Owner: the same copy enqueued on `stream` (host_ptr should be pinned); no synchronisation. */
LCGS_B200_API int lcgs_b200_peer_read_async(lcgs_b200_ctx* ctx, const void* dev_ptr, void* host_ptr, size_t bytes,
                                            lcgs_b200_stream stream);
LCGS_B200_API int lcgs_b200_peer_close(lcgs_b200_ctx* ctx, void* dev_ptr); /* unmap (other ranks) */
LCGS_B200_API int lcgs_b200_peer_free(lcgs_b200_ctx* ctx, void* dev_ptr);  /* free (owner) */

/* Device-side flow control for such a buffer: 32-bit sequence words that live in it (owner's memory) let a
 * writer tell the owner "slot s holds frame j" and the owner tell the writer "slot s may be overwritten",
 * entirely in stream order -- no host synchronisation and no collective between frames.
 *   signal: after everything enqueued before it on `stream` has completed (the frame's stores included), store
 *           `value` to *flag with system-scope release semantics (works through a peer mapping).
 *   wait:   hold `stream` until *flag >= value (system-scope acquire; one polling thread).  Gives up after
 *           timeout_ms (then sets the context's sticky flow-control error, see lcgs_b200_peer_error) so that a
 *           dead peer can never hang the GPU. */
LCGS_B200_API int lcgs_b200_peer_signal(lcgs_b200_ctx* ctx, uint32_t* flag, uint32_t value, lcgs_b200_stream stream);
LCGS_B200_API int lcgs_b200_peer_wait(lcgs_b200_ctx* ctx, const uint32_t* flag, uint32_t value, uint32_t timeout_ms,
                                      lcgs_b200_stream stream);
/* Synchronises the device; *timed_out = number of waits that gave up since the context was created. */
LCGS_B200_API int lcgs_b200_peer_error(lcgs_b200_ctx* ctx, uint32_t* timed_out);
/* The consumer's read of a delivered frame: *out (device memory, 8-byte aligned) = wrap-around sum of the `num_words`
 * 32-bit words at `data` (16-byte aligned), as one 64-bit integer -- exact and independent of the summation order. */
LCGS_B200_API int lcgs_b200_checksum_u32(lcgs_b200_ctx* ctx, const void* data, size_t num_words, uint64_t* out,
                                         lcgs_b200_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* LCGS_B200_H */
