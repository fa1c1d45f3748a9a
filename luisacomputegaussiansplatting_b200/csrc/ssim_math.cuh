// ssim_math.cuh -- the per-pixel arithmetic of the SSIM loss (lcgs_b200_ssim, ssim.cu): the window weights, and the
// SSIM value and its partials with respect to the three moments that involve the image, from the five moments.
//
// No reference counterpart: the reference renders only.  The semantics are those of the 3DGS training loss's ssim()
// (utils/loss_utils.py): an 11-tap Gaussian window of sigma 1.5, applied separably and per channel with zero padding
// of 5, C1 = 0.01^2, C2 = 0.03^2, the mean over channels and pixels.  Like lcgs_grad.cuh every function is
// __host__ __device__, so tests/ssim_mirror runs the same source on the CPU against torch autograd.
//
//   mx = G*x, my = G*y, exx = G*(x^2), eyy = G*(y^2), exy = G*(x y)
//   A = 2 mx my + C1,  B = 2 (exy - mx my) + C2,  Cc = mx^2 + my^2 + C1,  D = (exx - mx^2) + (eyy - my^2) + C2
//   s = A B / (Cc D)
//   P0 = ds/dmx  = 2 (my (B - A) + mx s (Cc - D)) / (Cc D)   (A, Cc, and through exx - mx^2, exy - mx my, B and D)
//   P1 = ds/dexx = -s / D
//   P2 = ds/dexy = 2 A / (Cc D)
//   dSSIM/dx_p = (1/N) ((G*P0)_p + 2 x_p (G*P1)_p + y_p (G*P2)_p),  N = 3 H W
// s is evaluated as (A / Cc) (B / D), and P0 in the factored form above, so that for x == y (A == Cc and B == D
// bit for bit) s is exactly 1 and P0 exactly 0.
#pragma once

#include "lcgs_math.cuh"

namespace lcgs_b200 {

constexpr int kSsimTaps = 11;
constexpr int kSsimRadius = 5;

// g_k = exp(-(k-5)^2 / 4.5) / sum_j exp(-(j-5)^2 / 4.5), each rounded once from double to float
#define LCGS_SSIM_WEIGHTS                                                                                             \
    { 1.028380124e-03f, 7.598758209e-03f, 3.600077331e-02f, 1.093606874e-01f, 2.130055428e-01f, 2.660117149e-01f,    \
      2.130055428e-01f, 1.093606874e-01f, 3.600077331e-02f, 7.598758209e-03f, 1.028380124e-03f }

LCGS_HD float ssim_weight(int k)
{
    const float w[kSsimTaps] = LCGS_SSIM_WEIGHTS;
    return w[k];
}

struct SsimPixel {
    float s;           // the pixel's SSIM
    float p0, p1, p2;  // ds/dmx, ds/dexx, ds/dexy
};

LCGS_HD SsimPixel ssim_pixel(float mx, float my, float exx, float eyy, float exy)
{
    const float C1 = (float)(0.01 * 0.01), C2 = (float)(0.03 * 0.03);
    const float mxy = mx * my, mxx = mx * mx, myy = my * my;
    const float A  = 2.0f * mxy + C1;
    const float B  = 2.0f * (exy - mxy) + C2;
    const float Cc = (mxx + myy) + C1;
    const float D  = ((exx - mxx) + (eyy - myy)) + C2;
    const float ra = A / Cc, rb = B / D, cd = Cc * D;
    SsimPixel   r;
    r.s  = ra * rb;
    r.p0 = 2.0f * (my * (B - A) + (mx * r.s) * (Cc - D)) / cd;
    r.p1 = -r.s / D;
    r.p2 = 2.0f * ra / D;
    return r;
}

}  // namespace lcgs_b200
