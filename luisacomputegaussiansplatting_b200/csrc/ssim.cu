// ssim.cu -- SSIM of a planar image against a reference, and its gradient with respect to the image (lcgs_b200_ssim).
// No reference counterpart: the reference renders only.  The per-pixel arithmetic and the semantics are in
// ssim_math.cuh.
//
//  * ssim_forward_kernel<GRAD> : one 256-thread CTA per 32x32 output tile and channel.  The tile's x and y plus a
//    5-pixel halo (42x42, zeros outside the image) are staged in shared memory with row-contiguous loads; the
//    horizontal 11-tap pass makes the five moments of the 42 rows, the vertical pass those of the 32x32 pixels, each
//    tap one FMA.  Every pixel's s joins the CTA's double partial sum (shuffles, then the eight warps in a fixed
//    order), written to the context's ssim_ws.  GRAD: the three partial maps P0..P2 of the pixel go to ssim_ws too
//    ([3 maps][3 channels][H][W], 36 B per pixel).
//  * ssim_reduce_kernel : one CTA sums the per-CTA partials in double in a fixed order and writes the mean.
//  * ssim_backward_kernel : the same tiling over the partial maps (zeros outside the image, so the transposed filter is
//    the same zero-padded one): d_p = (1/N) ((G*P0)_p + 2 x_p (G*P1)_p + y_p (G*P2)_p).  Launched only when the
//    gradient is requested.
// No atomics: the value and the gradient are the same bits from run to run.
#include "common.cuh"
#include "ssim_math.cuh"

namespace lcgs_b200 {

constexpr int kSsimTile    = 32;                             // output tile edge
constexpr int kSsimHalo    = kSsimTile + 2 * kSsimRadius;    // staged window edge
constexpr int kSsimThreads = 256;
constexpr int kSsimRowStep = kSsimThreads / kSsimTile;       // rows apart of one thread's pixels in the vertical pass
constexpr int kSsimReduceThreads = 512;

struct SsimArgs {
    int          W, H;
    uint32_t     gx;     // tiles per row
    size_t       plane;  // W * H
    const float* x;      // [3][H][W] image
    const float* y;      // [3][H][W] reference
    float*       maps;   // [3][3][H][W] P0, P1, P2 per channel
    double*      partials;
};

// (kSsimHalo x kSsimHalo) window of one channel plane at (x0 - 5, y0 - 5); zero outside the image
__device__ __forceinline__ void ssim_stage(float (*dst)[kSsimHalo], const float* __restrict__ src, int W, int H, int x0, int y0)
{
    for (int i = threadIdx.x; i < kSsimHalo * kSsimHalo; i += kSsimThreads) {
        const int r = i / kSsimHalo, c = i - r * kSsimHalo;
        const int gx = x0 - kSsimRadius + c, gy = y0 - kSsimRadius + r;
        dst[r][c] = (gx >= 0 && gx < W && gy >= 0 && gy < H) ? __ldg(src + (size_t)gy * W + gx) : 0.0f;
    }
}

__device__ __forceinline__ void ssim_tile_origin(const SsimArgs& a, int* x0, int* y0)
{
    const uint32_t ty = blockIdx.x / a.gx;
    *x0 = (int)(blockIdx.x - ty * a.gx) * kSsimTile;
    *y0 = (int)ty * kSsimTile;
}

template <bool GRAD>
__global__ void __launch_bounds__(kSsimThreads) ssim_forward_kernel(const SsimArgs a)
{
    __shared__ float  s_x[kSsimHalo][kSsimHalo], s_y[kSsimHalo][kSsimHalo];
    __shared__ float  s_h[5][kSsimHalo][kSsimTile];  // horizontally filtered mx, my, exx, eyy, exy
    __shared__ double s_warp[kSsimThreads / 32];
    const int    ch = blockIdx.y;
    const size_t co = (size_t)ch * a.plane;
    int          x0, y0;
    ssim_tile_origin(a, &x0, &y0);
    ssim_stage(s_x, a.x + co, a.W, a.H, x0, y0);
    ssim_stage(s_y, a.y + co, a.W, a.H, x0, y0);
    __syncthreads();

    for (int i = threadIdx.x; i < kSsimHalo * kSsimTile; i += kSsimThreads) {
        const int r = i / kSsimTile, c = i % kSsimTile;
        float     mx = 0.f, my = 0.f, exx = 0.f, eyy = 0.f, exy = 0.f;
#pragma unroll
        for (int k = 0; k < kSsimTaps; k++) {
            const float w = ssim_weight(k), xv = s_x[r][c + k], yv = s_y[r][c + k];
            mx  = __fmaf_rn(w, xv, mx);
            my  = __fmaf_rn(w, yv, my);
            exx = __fmaf_rn(w, xv * xv, exx);
            eyy = __fmaf_rn(w, yv * yv, eyy);
            exy = __fmaf_rn(w, xv * yv, exy);
        }
        s_h[0][r][c] = mx; s_h[1][r][c] = my; s_h[2][r][c] = exx; s_h[3][r][c] = eyy; s_h[4][r][c] = exy;
    }
    __syncthreads();

    const int c = threadIdx.x % kSsimTile, px = x0 + c;
    double    sum = 0.0;
#pragma unroll 1
    for (int r = threadIdx.x / kSsimTile; r < kSsimTile; r += kSsimRowStep) {
        const int py = y0 + r;
        if (px >= a.W || py >= a.H) continue;
        float m[5] = { 0.f, 0.f, 0.f, 0.f, 0.f };
#pragma unroll
        for (int k = 0; k < kSsimTaps; k++) {
            const float w = ssim_weight(k);
#pragma unroll
            for (int j = 0; j < 5; j++) m[j] = __fmaf_rn(w, s_h[j][r + k][c], m[j]);
        }
        const SsimPixel p = ssim_pixel(m[0], m[1], m[2], m[3], m[4]);
        sum += (double)p.s;
        if (GRAD) {
            const size_t q = (size_t)py * a.W + px;
            a.maps[(size_t)(0 * 3 + ch) * a.plane + q] = p.p0;
            a.maps[(size_t)(1 * 3 + ch) * a.plane + q] = p.p1;
            a.maps[(size_t)(2 * 3 + ch) * a.plane + q] = p.p2;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = sum;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < kSsimThreads / 32; w++) t += s_warp[w];
        a.partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = t;
    }
}

// Sums the n partials in a fixed order (strided per thread, then a fixed tree) and writes their mean over N pixels.
__global__ void __launch_bounds__(kSsimReduceThreads)
    ssim_reduce_kernel(const double* __restrict__ partials, uint32_t n, double N, float* __restrict__ ssim)
{
    __shared__ double s[kSsimReduceThreads];
    double            acc = 0.0;
    for (uint32_t j = threadIdx.x; j < n; j += kSsimReduceThreads) acc += partials[j];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int w = kSsimReduceThreads / 2; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) s[threadIdx.x] += s[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) *ssim = (float)(s[0] / N);
}

__global__ void __launch_bounds__(kSsimThreads) ssim_backward_kernel(const SsimArgs a, float inv_n, float* __restrict__ grad)
{
    __shared__ float s_p[3][kSsimHalo][kSsimHalo];
    __shared__ float s_h[3][kSsimHalo][kSsimTile];
    const int    ch = blockIdx.y;
    const size_t co = (size_t)ch * a.plane;
    int          x0, y0;
    ssim_tile_origin(a, &x0, &y0);
#pragma unroll
    for (int m = 0; m < 3; m++) ssim_stage(s_p[m], a.maps + (size_t)(m * 3 + ch) * a.plane, a.W, a.H, x0, y0);
    __syncthreads();

    for (int i = threadIdx.x; i < kSsimHalo * kSsimTile; i += kSsimThreads) {
        const int r = i / kSsimTile, c = i % kSsimTile;
        float     f[3] = { 0.f, 0.f, 0.f };
#pragma unroll
        for (int k = 0; k < kSsimTaps; k++) {
            const float w = ssim_weight(k);
#pragma unroll
            for (int m = 0; m < 3; m++) f[m] = __fmaf_rn(w, s_p[m][r][c + k], f[m]);
        }
#pragma unroll
        for (int m = 0; m < 3; m++) s_h[m][r][c] = f[m];
    }
    __syncthreads();

    const int c = threadIdx.x % kSsimTile, px = x0 + c;
#pragma unroll 1
    for (int r = threadIdx.x / kSsimTile; r < kSsimTile; r += kSsimRowStep) {
        const int py = y0 + r;
        if (px >= a.W || py >= a.H) continue;
        float f[3] = { 0.f, 0.f, 0.f };
#pragma unroll
        for (int k = 0; k < kSsimTaps; k++) {
            const float w = ssim_weight(k);
#pragma unroll
            for (int m = 0; m < 3; m++) f[m] = __fmaf_rn(w, s_h[m][r + k][c], f[m]);
        }
        const size_t q  = co + (size_t)py * a.W + px;
        const float  xv = __ldg(a.x + q), yv = __ldg(a.y + q);
        grad[q] = __fmaf_rn(2.0f * xv, f[1], __fmaf_rn(yv, f[2], f[0])) * inv_n;
    }
}

int launch_ssim(lcgs_b200_ctx* ctx, int W, int H, const float* img, const float* ref, float* ssim, float* grad,
                cudaStream_t s)
{
    SsimArgs a;
    a.W = W; a.H = H;
    a.gx    = (uint32_t)((W + kSsimTile - 1) / kSsimTile);
    a.plane = (size_t)W * H;
    a.x = img; a.y = ref;
    const uint32_t tiles     = a.gx * (uint32_t)((H + kSsimTile - 1) / kSsimTile);
    const size_t   map_bytes = grad ? ((9 * a.plane * sizeof(float) + 255) & ~(size_t)255) : 0;
    int            rc;
    if ((rc = ws_reserve(ctx, ctx->ssim_ws, map_bytes + (size_t)3 * tiles * sizeof(double)))) return rc;
    a.maps     = (float*)ctx->ssim_ws.ptr;
    a.partials = (double*)((char*)ctx->ssim_ws.ptr + map_bytes);
    const dim3 grid(tiles, 3);
    if (grad)
        ssim_forward_kernel<true><<<grid, kSsimThreads, 0, s>>>(a);
    else
        ssim_forward_kernel<false><<<grid, kSsimThreads, 0, s>>>(a);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    const double N = 3.0 * (double)a.plane;
    ssim_reduce_kernel<<<1, kSsimReduceThreads, 0, s>>>(a.partials, 3 * tiles, N, ssim);
    LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    if (grad) {
        ssim_backward_kernel<<<grid, kSsimThreads, 0, s>>>(a, (float)(1.0 / N), grad);
        LCGS_CUDA_CHECK(ctx, cudaGetLastError());
    }
    return LCGS_B200_OK;
}

}  // namespace lcgs_b200
