// lcgs_grad.cuh -- derivatives of the forward splat path (lcgs_math.cuh), per blended pair and per Gaussian.
//
// No reference counterpart: the reference renders only (its util/sh.hpp carries unfinished, never-called SH
// backward helpers).  Like lcgs_math.cuh every function is __host__ __device__, so tests/grad_mirror runs the very
// same source on the CPU against torch autograd before any GPU time is spent.
//
// Semantics (derived from the forward as written; L is a scalar loss of the planar image, G = dL/dC of a pixel):
//   blend, per pixel, over the entries i = 1..n the forward blended, in list order:
//     w_i = T_i alpha_i,  T_{i+1} = T_i (1 - alpha_i),  C = sum w_i c_i + T_{n+1} bg
//     dL/dc_i     = w_i G
//     dL/dalpha_i = T_i (c_i . G) - (R_i . G) / (1 - alpha_i),   R_i = C - sum_{j<=i} w_j c_j
//   C is the forward's own pixel value, so the walk runs front to back like the forward, with its culling, its
//   alpha test and its T (1 - alpha) < 1e-4 stop; entries the alpha test rejects and the entry that would saturate
//   the pixel get no gradient.
//   alpha = min(0.99, o e^power): zero gradient where the cap is active, else dalpha/do = alpha / o and
//   dalpha/dpower = alpha; power = -1/2 (A dx^2 + C dy^2) - B dx dy with dx = mu_x - x_p, dy = mu_y - y_p (Q2).
//   The blend accumulates dL/dpower = dL/dalpha * alpha, which is also dL/dlog(o): the opacity gradient is that sum
//   divided by o.
//   preprocess: view_transform, ewa_cov2d (unnormalised quaternion, scale_modifier, the tx/ty clamp to
//   +-1.3 tanfov: gradient only where the clamp is inactive), splat_from_cov (the +0.3 low-pass and det + 1e-6) and
//   sh_color (the view direction of degree >= 1 reaches pos; the [0,1] colour clamp passes gradient per channel only
//   where it is inactive) are differentiated exactly as written.  radius, the tile rect, depth order and
//   tiles_touched are discrete.
//   aux planes (the blend's optional alpha and depth planes, A = 1 - T_{n+1} and D = sum w_i z_i): two more channels
//   with colours 1 and z_i and a background of 0 (see PixelGradAux); depth z = view z, so dL/dz joins dL/dvz in
//   project_backward.
//   camera pose (project_backward_pose, preprocess_pose_grad_kernel): V = vp.view, column-major, p_view[k] =
//   sum_c V[c*4+k] p[c] + V[12+k].  With dv = dL/dp_view (dL/dz of the depth plane included) and the EWA Jacobian's
//   T0 = J00 V_col0 + J02 V_col2, T1 = J11 V_col1 + J12 V_col2 (rows r of mat3(view)):
//     dL/dV[c*4+k] = dv[k] p[c] (c < 3),  dL/dV[12+k] = dv[k],
//     dL/dV[r*4+0] += J00 dT0[r],  dL/dV[r*4+1] += J11 dT1[r],  dL/dV[r*4+2] += J02 dT0[r] + J12 dT1[r];
//   V[3], V[7], V[11], V[15] never enter the forward.  dL/dcam_pos = -(sh_color's view-direction term of dL/dpos),
//   zero for degree 0 and where every colour channel is clamped.  proj, focal and tanfov are held fixed.
#pragma once

#include "lcgs_math.cuh"

namespace lcgs_b200 {

// Packed per-Gaussian gradient of the blend's inputs: 12 floats = three float4, so the blend backward can accumulate
// it with vector reductions.  kG2LogOp holds dL/dpower summed over the Gaussian's pairs (= dL/dlog(opacity)).
// kG2Depth holds dL/d(view depth) from the depth plane; only the aux blend backward writes it (kGrad2DAuxValues), the
// image-only one leaves it at 0.
enum {
    kG2MeanX = 0, kG2MeanY, kG2Conic0, kG2Conic1, kG2Conic2, kG2LogOp, kG2Red, kG2Green, kG2Blue, kG2Depth,
    kGrad2DValues = 9, kGrad2DAuxValues = 10, kGrad2DFloats = 12
};

// Per-pixel state of the backward walk.  T < 0 marks a finished pixel (saturated or outside the image), as in the
// forward.  CG = C . G of the finished pixel; SG = sum_{j<=i} w_j (c_j . G) so far, so that R_i . G = CG - SG.
struct PixelGrad {
    float T, CG, SG;
    float G[3];
};

LCGS_HD PixelGrad pixel_grad_init(bool inside, const float* C, const float* G)
{
    PixelGrad p;
    p.T  = inside ? 1.0f : -1.0f;
    p.CG = (C[0] * G[0] + C[1] * G[1]) + C[2] * G[2];
    p.SG = 0.0f;
    p.G[0] = G[0]; p.G[1] = G[1]; p.G[2] = G[2];
    return p;
}

// The aux planes are two more channels of the same blend with a background of 0: the alpha plane A = 1 - T has colour
// 1 for every entry, the depth plane D = sum w_i z_i has colour z_i = depth[id].  With GA = dL/dA and GD = dL/dD the
// per-entry colour dot product becomes c_i . G + z_i GD + GA and the final one C . G + D GD + A GA, so the aux walk is
// the colour walk with that 5-channel dot product, plus dL/dz_i = w_i GD.
struct PixelGradAux {
    PixelGrad p;  // p.CG includes the planes' terms
    float     GA, GD;
};

LCGS_HD PixelGradAux pixel_grad_aux_init(bool inside, const float* C, const float* G, float A, float D, float GA, float GD)
{
    PixelGradAux q;
    q.p    = pixel_grad_init(inside, C, G);
    q.p.CG = (q.p.CG + D * GD) + A * GA;
    q.GA   = GA;
    q.GD   = GD;
    return q;
}

// One entry of the pixel's front-to-back walk (AUX: with the aux channels, z = the entry's view depth).
template <bool AUX>
LCGS_HD bool blend_entry_grad_t(PixelGrad& px, bool ok, float alpha_raw, float dx, float dy, float a, float b, float c,
                                const float* rgb, float z, float GA, float GD, float* g)
{
    if (!ok || !(px.T > 0.0f)) return false;
    const float T      = px.T;
    const float alpha  = fminf(0.99f, alpha_raw);
    const float test_T = T * (1.0f - alpha);
    if (test_T < 0.0001f) {  // saturates: not blended, and the pixel is finished
        px.T = -T;
        return false;
    }
    const float w  = T * alpha;
    float       cG = (rgb[0] * px.G[0] + rgb[1] * px.G[1]) + rgb[2] * px.G[2];
    if constexpr (AUX) cG = (cG + z * GD) + GA;
    px.SG              = px.SG + w * cG;
    const float dalpha = T * cG - (px.CG - px.SG) / (1.0f - alpha);
    const float gp     = alpha_raw < 0.99f ? dalpha * alpha : 0.0f;  // dL/dpower; zero under the cap
    g[kG2MeanX]  += gp * ((2.0f * a) * dx + b * dy);
    g[kG2MeanY]  += gp * ((2.0f * c) * dy + b * dx);
    g[kG2Conic0] += gp * (-0.5f * (dx * dx));
    g[kG2Conic1] += gp * (-(dx * dy));
    g[kG2Conic2] += gp * (-0.5f * (dy * dy));
    g[kG2LogOp]  += gp;
    g[kG2Red]    += w * px.G[0];
    g[kG2Green]  += w * px.G[1];
    g[kG2Blue]   += w * px.G[2];
    if constexpr (AUX) g[kG2Depth] += w * GD;
    px.T = test_T;
    return true;
}

// One entry of the pixel's front-to-back walk.  ok = the entry passed the alpha test (power <= 0 and power >= the
// Gaussian's threshold); alpha_raw = o e^power as the forward evaluated it, before the 0.99 cap.  (a, b, c) are the
// record's pre-scaled conic (-0.5 conic.x, -conic.y, -0.5 conic.z), (dx, dy) = mean - pixel.  Adds the pair's
// contribution to g[kGrad2DValues] and returns true iff the forward blended the entry.  T is updated with the
// forward's own operations, so the walk stops exactly where the forward's did.
LCGS_HD bool blend_entry_grad(PixelGrad& px, bool ok, float alpha_raw, float dx, float dy, float a, float b, float c,
                              const float* rgb, float* g)
{
    return blend_entry_grad_t<false>(px, ok, alpha_raw, dx, dy, a, b, c, rgb, 0.0f, 0.0f, 0.0f, g);
}

// The same step on the aux channels: adds to g[kGrad2DAuxValues] (kG2Depth += w GD).
LCGS_HD bool blend_entry_grad_aux(PixelGradAux& px, bool ok, float alpha_raw, float dx, float dy, float a, float b,
                                  float c, const float* rgb, float z, float* g)
{
    return blend_entry_grad_t<true>(px.p, ok, alpha_raw, dx, dy, a, b, c, rgb, z, px.GA, px.GD, g);
}

// ---------------------------------------------------------------------------------------------
// sh_color backward.  dcol = dL/d(post-clamp colour); adds dL/dpos of the view direction into dpos and writes every
// coefficient's gradient through dsh(k, c, value) (k < (deg+1)^2).  Recomputes the pre-clamp colour with the
// forward's operations, so the clamp decision is the forward's.
// ---------------------------------------------------------------------------------------------
template <typename ShIn, typename ShOut>
LCGS_HD void sh_color_backward(int deg, const float* cam_pos, float px, float py, float pz, const ShIn& sh,
                               const float* dcol, const ShOut& dsh, float* dpos)
{
    float x = 0.f, y = 0.f, z = 0.f, inv = 0.f;
    if (deg > 0) {
        const float dx = px - cam_pos[0], dy = py - cam_pos[1], dz = pz - cam_pos[2];
        const float len2 = (dx * dx + dy * dy) + dz * dz;
        inv = 1.0f / sqrtf(len2);
        x = dx * inv; y = dy * inv; z = dz * inv;
    }
    float dres[3];
    {
        // sh_color's sum before the clamp, in the forward's order
        float r[3] = { sh(0, 0) * LCGS_SH_C0, sh(0, 1) * LCGS_SH_C0, sh(0, 2) * LCGS_SH_C0 };
        if (deg > 0) {
#pragma unroll
            for (int c = 0; c < 3; c++) r[c] = r[c] + (-LCGS_SH_C1) * ((sh(1, c) * y - sh(2, c) * z) + sh(3, c) * x);
            if (deg > 1) {
                const float xx = x * x, yy = y * y, yz = y * z, zz = z * z, zx = z * x, xy = x * y;
                const float k0 = 1.0925484305920792f * xy;
                const float k1 = -1.0925484305920792f * yz;
                const float k2 = 0.31539156525252005f * ((2.0f * zz - xx) - yy);
                const float k3 = -1.0925484305920792f * zx;
                const float k4 = 0.5462742152960396f * (xx - yy);
#pragma unroll
                for (int c = 0; c < 3; c++)
                    r[c] = r[c] + ((((k0 * sh(4, c) + k1 * sh(5, c)) + k2 * sh(6, c)) + k3 * sh(7, c)) + k4 * sh(8, c));
                if (deg > 2) {
                    const float m0 = -0.5900435899266435f * y * (3.0f * xx - yy);
                    const float m1 = 2.890611442640554f * xy * z;
                    const float m2 = -0.4570457994644658f * y * ((4.0f * zz - xx) - yy);
                    const float m3 = 0.3731763325901154f * z * ((2.0f * zz - 3.0f * xx) - 3.0f * yy);
                    const float m4 = -0.4570457994644658f * x * ((4.0f * zz - xx) - yy);
                    const float m5 = 1.445305721320277f * z * (xx - yy);
                    const float m6 = -0.5900435899266435f * x * (xx - 3.0f * yy);
#pragma unroll
                    for (int c = 0; c < 3; c++)
                        r[c] = r[c] + ((((((m0 * sh(9, c) + m1 * sh(10, c)) + m2 * sh(11, c)) + m3 * sh(12, c)) + m4 * sh(13, c)) +
                                        m5 * sh(14, c)) +
                                       m6 * sh(15, c));
                }
            }
        }
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const float v = r[c] + 0.5f;
            dres[c]       = (v >= 0.0f && v <= 1.0f) ? dcol[c] : 0.0f;  // the clamp passes gradient where inactive
        }
    }
#pragma unroll
    for (int c = 0; c < 3; c++) dsh(0, c, LCGS_SH_C0 * dres[c]);
    if (deg < 1) return;
    float gx = 0.f, gy = 0.f, gz = 0.f;  // dL/d(normalised direction)
#pragma unroll
    for (int c = 0; c < 3; c++) {
        dsh(1, c, -LCGS_SH_C1 * y * dres[c]);
        dsh(2, c, LCGS_SH_C1 * z * dres[c]);
        dsh(3, c, -LCGS_SH_C1 * x * dres[c]);
        gx += -LCGS_SH_C1 * sh(3, c) * dres[c];
        gy += -LCGS_SH_C1 * sh(1, c) * dres[c];
        gz += LCGS_SH_C1 * sh(2, c) * dres[c];
    }
    if (deg > 1) {
        const float K = 1.0925484305920792f, Q = 0.31539156525252005f, Hh = 0.5462742152960396f;
        const float xx = x * x, yy = y * y, zz = z * z;
        const float k[5] = { K * (x * y), -K * (y * z), Q * ((2.0f * zz - xx) - yy), -K * (z * x), Hh * (xx - yy) };
        // d k_j / d(x, y, z)
        const float kx[5] = { K * y, 0.0f, -2.0f * Q * x, -K * z, 2.0f * Hh * x };
        const float ky[5] = { K * x, -K * z, -2.0f * Q * y, 0.0f, -2.0f * Hh * y };
        const float kz[5] = { 0.0f, -K * y, 4.0f * Q * z, -K * x, 0.0f };
#pragma unroll
        for (int c = 0; c < 3; c++)
#pragma unroll
            for (int j = 0; j < 5; j++) {
                dsh(4 + j, c, k[j] * dres[c]);
                const float s = sh(4 + j, c) * dres[c];
                gx += kx[j] * s; gy += ky[j] * s; gz += kz[j] * s;
            }
        if (deg > 2) {
            const float A = -0.5900435899266435f, B = 2.890611442640554f, Cc = -0.4570457994644658f;
            const float D = 0.3731763325901154f, E = 1.445305721320277f;
            const float m[7] = { A * y * (3.0f * xx - yy), B * (x * y) * z, Cc * y * ((4.0f * zz - xx) - yy),
                                 D * z * ((2.0f * zz - 3.0f * xx) - 3.0f * yy), Cc * x * ((4.0f * zz - xx) - yy),
                                 E * z * (xx - yy), A * x * (xx - 3.0f * yy) };
            const float mx[7] = { 6.0f * A * x * y, B * y * z, -2.0f * Cc * x * y, -6.0f * D * x * z,
                                  Cc * ((4.0f * zz - 3.0f * xx) - yy), 2.0f * E * x * z, A * (3.0f * xx - 3.0f * yy) };
            const float my[7] = { A * (3.0f * xx - 3.0f * yy), B * x * z, Cc * ((4.0f * zz - xx) - 3.0f * yy), -6.0f * D * y * z,
                                  -2.0f * Cc * x * y, -2.0f * E * y * z, -6.0f * A * x * y };
            const float mz[7] = { 0.0f, B * x * y, 8.0f * Cc * y * z, D * ((6.0f * zz - 3.0f * xx) - 3.0f * yy),
                                  8.0f * Cc * x * z, E * (xx - yy), 0.0f };
#pragma unroll
            for (int c = 0; c < 3; c++)
#pragma unroll
                for (int j = 0; j < 7; j++) {
                    dsh(9 + j, c, m[j] * dres[c]);
                    const float s = sh(9 + j, c) * dres[c];
                    gx += mx[j] * s; gy += my[j] * s; gz += mz[j] * s;
                }
        }
    }
    // through the normalisation: d(d/|d|) = (g - n (n . g)) / |d|
    const float ng = (x * gx + y * gy) + z * gz;
    dpos[0] += (gx - x * ng) * inv;
    dpos[1] += (gy - y * ng) * inv;
    dpos[2] += (gz - z * ng) * inv;
}

// ---------------------------------------------------------------------------------------------
// Projection backward: from the packed 2D gradient g2 (pixel mean, conic) of one visible Gaussian to dL/dpos,
// dL/dscale and dL/drotq (stored order r, x, y, z).  dpos is accumulated into (the SH term adds to it too), dscale
// and drot are written.  POSE: dL/d(view) is accumulated into dview[12], dview[c*3+k] for V[c*4+k] (k < 3).
// ---------------------------------------------------------------------------------------------
template <bool POSE>
LCGS_HD void project_backward_t(const ViewParams& vp, float scale_modifier, float px, float py, float pz, float s0,
                                float s1, float s2, float qr, float qx, float qy, float qz, const float* g2, float* dpos,
                                float* dscale, float* drot, float* dview)
{
    const ViewPoint pv = view_transform(vp, px, py, pz);
    // ---- forward intermediates, as ewa_cov2d computes them
    const float sc[3] = { scale_modifier * s0, scale_modifier * s1, scale_modifier * s2 };
    const float x = qx, y = qy, z = qz, w = qr;
    float       R[3][3];
    R[0][0] = (1.0f - (2.0f * y) * y) - (2.0f * z) * z;
    R[0][1] = (2.0f * x) * y + (2.0f * z) * w;
    R[0][2] = (2.0f * x) * z - (2.0f * y) * w;
    R[1][0] = (2.0f * x) * y - (2.0f * z) * w;
    R[1][1] = (1.0f - (2.0f * x) * x) - (2.0f * z) * z;
    R[1][2] = (2.0f * y) * z + (2.0f * x) * w;
    R[2][0] = (2.0f * x) * z + (2.0f * y) * w;
    R[2][1] = (2.0f * y) * z - (2.0f * x) * w;
    R[2][2] = (1.0f - (2.0f * x) * x) - (2.0f * y) * y;
    float M[3][3];
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
        for (int r = 0; r < 3; r++) M[c][r] = sc[c] * R[c][r];
    float Sg[3][3];
#pragma unroll
    for (int c = 0; c < 3; c++)
#pragma unroll
        for (int r = 0; r < 3; r++) Sg[c][r] = (M[0][c] * M[0][r] + M[1][c] * M[1][r]) + M[2][c] * M[2][r];
    const float limx = 1.3f * vp.tanfovx, limy = 1.3f * vp.tanfovy;
    const float txtz = pv.x / pv.z, tytz = pv.y / pv.z;
    const float ctx = clampf(txtz, -limx, limx), cty = clampf(tytz, -limy, limy);
    const float tx = ctx * pv.z, ty = cty * pv.z, tz = pv.z;
    const float J00 = vp.focalx / tz, J11 = vp.focaly / tz;
    const float J02 = (-vp.focalx * tx) / (tz * tz), J12 = (-vp.focaly * ty) / (tz * tz);
    const float* V = vp.view;
    float        T0[3], T1[3];
#pragma unroll
    for (int r = 0; r < 3; r++) {
        T0[r] = J00 * V[r * 4 + 0] + J02 * V[r * 4 + 2];
        T1[r] = J11 * V[r * 4 + 1] + J12 * V[r * 4 + 2];
    }
    float cov[3];
    {
        float A[3][2];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            A[c][0] = (Sg[c][0] * T0[0] + Sg[c][1] * T0[1]) + Sg[c][2] * T0[2];
            A[c][1] = (Sg[c][0] * T1[0] + Sg[c][1] * T1[1]) + Sg[c][2] * T1[2];
        }
        cov[0] = (T0[0] * A[0][0] + T0[1] * A[1][0]) + T0[2] * A[2][0];
        cov[1] = (T0[0] * A[0][1] + T0[1] * A[1][1]) + T0[2] * A[2][1];
        cov[2] = (T1[0] * A[0][1] + T1[1] * A[1][1]) + T1[2] * A[2][1];
    }

    // ---- conic = inverse of the low-passed covariance (splat_from_cov)
    const float a = cov[0] + 0.3f, b = cov[1], c = cov[2] + 0.3f;
    const float det = a * c - b * b;
    const float inv = 1.0f / (det + 1e-6f);
    const float g0 = g2[kG2Conic0], g1 = g2[kG2Conic1], gc2 = g2[kG2Conic2];
    // d(inv * adj)/d(a, b, c) written in the conic entries k = (inv c, -inv b, inv a) themselves: the same value as
    // the chain through det, without its cancellation (g inv - g inv^2 a c) for thin Gaussians; e = 1e-6 inv^2
    const float k0 = inv * c, k1 = inv * (-b), k2 = inv * a, e = 1e-6f * (inv * inv);
    const float dc0 = ((-g0 * (k0 * k0) - g1 * (k0 * k1)) - gc2 * (k1 * k1)) + gc2 * e;                 // dL/dcov[0]
    const float dc1 = (-2.0f * g0 * (k0 * k1) - g1 * ((k0 * k2 + k1 * k1) + e)) - 2.0f * gc2 * (k1 * k2);  // dL/dcov[1]
    const float dc2 = ((-g0 * (k1 * k1) - g1 * (k1 * k2)) - gc2 * (k2 * k2)) + g0 * e;                 // dL/dcov[2]

    // ---- cov = (T0' S T0, T0' S T1, T1' S T1)
    float dS[3][3], dT0[3], dT1[3];
#pragma unroll
    for (int i = 0; i < 3; i++) {
#pragma unroll
        for (int j = 0; j < 3; j++) dS[i][j] = (dc0 * T0[i]) * T0[j] + (dc1 * T0[i]) * T1[j] + (dc2 * T1[i]) * T1[j];
        const float s_t0 = (Sg[i][0] * T0[0] + Sg[i][1] * T0[1]) + Sg[i][2] * T0[2];  // (S T0)_i
        const float t0_s = (T0[0] * Sg[0][i] + T0[1] * Sg[1][i]) + T0[2] * Sg[2][i];  // (T0' S)_i
        const float s_t1 = (Sg[i][0] * T1[0] + Sg[i][1] * T1[1]) + Sg[i][2] * T1[2];
        const float t1_s = (T1[0] * Sg[0][i] + T1[1] * Sg[1][i]) + T1[2] * Sg[2][i];
        dT0[i] = dc0 * (s_t0 + t0_s) + dc1 * s_t1;
        dT1[i] = dc1 * t0_s + dc2 * (s_t1 + t1_s);
    }
    // S[c][r] = sum_k M[k][c] M[k][r]
    float dM[3][3];
#pragma unroll
    for (int k = 0; k < 3; k++)
#pragma unroll
        for (int j = 0; j < 3; j++) {
            float acc = 0.0f;
#pragma unroll
            for (int r = 0; r < 3; r++) acc += dS[j][r] * M[k][r] + dS[r][j] * M[k][r];
            dM[k][j] = acc;
        }
    float dR[3][3];
#pragma unroll
    for (int k = 0; k < 3; k++) {
        const float dsc = (dM[k][0] * R[k][0] + dM[k][1] * R[k][1]) + dM[k][2] * R[k][2];
        dscale[k]       = scale_modifier * dsc;
#pragma unroll
        for (int j = 0; j < 3; j++) dR[k][j] = dM[k][j] * sc[k];
    }
    const float dw = 2.0f * (((z * dR[0][1] - y * dR[0][2]) - z * dR[1][0]) + ((x * dR[1][2] + y * dR[2][0]) - x * dR[2][1]));
    const float dx = 2.0f * ((y * dR[0][1] + z * dR[0][2]) + (y * dR[1][0] - 2.0f * x * dR[1][1]) + (w * dR[1][2] + z * dR[2][0]) +
                             (-w * dR[2][1] - 2.0f * x * dR[2][2]));
    const float dy = 2.0f * ((-2.0f * y * dR[0][0] + x * dR[0][1]) + (-w * dR[0][2] + x * dR[1][0]) + (z * dR[1][2] + w * dR[2][0]) +
                             (z * dR[2][1] - 2.0f * y * dR[2][2]));
    const float dz = 2.0f * ((-2.0f * z * dR[0][0] + w * dR[0][1]) + (x * dR[0][2] - w * dR[1][0]) +
                             (-2.0f * z * dR[1][1] + y * dR[1][2]) + (x * dR[2][0] + y * dR[2][1]));
    drot[0] = dw; drot[1] = dx; drot[2] = dy; drot[3] = dz;

    // ---- T0 = J00 V_col0 + J02 V_col2, T1 = J11 V_col1 + J12 V_col2 (rows r of mat3(view))
    float dJ00 = 0.f, dJ02 = 0.f, dJ11 = 0.f, dJ12 = 0.f;
#pragma unroll
    for (int r = 0; r < 3; r++) {
        dJ00 += dT0[r] * V[r * 4 + 0];
        dJ02 += dT0[r] * V[r * 4 + 2];
        dJ11 += dT1[r] * V[r * 4 + 1];
        dJ12 += dT1[r] * V[r * 4 + 2];
    }
    const float tz2 = tz * tz, tz3 = tz2 * tz;
    const float dtx = dJ02 * (-vp.focalx) / tz2, dty = dJ12 * (-vp.focaly) / tz2;
    float dvz = -dJ00 * vp.focalx / tz2 - dJ11 * vp.focaly / tz2 + dJ02 * (2.0f * vp.focalx * tx) / tz3 +
                dJ12 * (2.0f * vp.focaly * ty) / tz3;
    float dvx = 0.f, dvy = 0.f;
    // tx = clamp(x / z) * z: the clamp passes gradient where it is inactive
    dvz += dtx * ctx + dty * cty;
    if (txtz >= -limx && txtz <= limx) {
        const float dq = dtx * pv.z;
        dvx += dq / pv.z;
        dvz += -dq * pv.x / (pv.z * pv.z);
    }
    if (tytz >= -limy && tytz <= limy) {
        const float dq = dty * pv.z;
        dvy += dq / pv.z;
        dvz += -dq * pv.y / (pv.z * pv.z);
    }
    // ---- the depth plane's part: depth = view z
    dvz += g2[kG2Depth];
    // ---- pixel mean: px = ((ndc + 1) W - 1) / 2, ndc = (v * proj) / (z + 1e-6)
    const float dndx = g2[kG2MeanX] * (0.5f * (float)(uint32_t)vp.width);
    const float dndy = g2[kG2MeanY] * (0.5f * (float)(uint32_t)vp.height);
    const float p_w  = 1.0f / (pv.z + 1e-6f);
    dvx += dndx * vp.proj[0] * p_w;
    dvy += dndy * vp.proj[5] * p_w;
    dvz += -((dndx * (pv.x * vp.proj[0]) + dndy * (pv.y * vp.proj[5])) * (p_w * p_w));
    // ---- view transform
    dpos[0] += (dvx * V[0] + dvy * V[1]) + dvz * V[2];
    dpos[1] += (dvx * V[4] + dvy * V[5]) + dvz * V[6];
    dpos[2] += (dvx * V[8] + dvy * V[9]) + dvz * V[10];
    if constexpr (POSE) {
        // the affine map p_view = mat3(view) p + view[12..14]
        const float dv[3] = { dvx, dvy, dvz }, p[3] = { px, py, pz };
#pragma unroll
        for (int k = 0; k < 3; k++) {
#pragma unroll
            for (int c = 0; c < 3; c++) dview[c * 3 + k] += dv[k] * p[c];
            dview[9 + k] += dv[k];
        }
        // the rows of mat3(view) in T0 and T1
#pragma unroll
        for (int r = 0; r < 3; r++) {
            dview[r * 3 + 0] += J00 * dT0[r];
            dview[r * 3 + 1] += J11 * dT1[r];
            dview[r * 3 + 2] += J02 * dT0[r] + J12 * dT1[r];
        }
    }
}

LCGS_HD void project_backward(const ViewParams& vp, float scale_modifier, float px, float py, float pz, float s0, float s1,
                              float s2, float qr, float qx, float qy, float qz, const float* g2, float* dpos, float* dscale,
                              float* drot)
{
    project_backward_t<false>(vp, scale_modifier, px, py, pz, s0, s1, s2, qr, qx, qy, qz, g2, dpos, dscale, drot, nullptr);
}

// project_backward that also accumulates dL/d(view) into dview[12] (dview[c*3+k] for vp.view[c*4+k], k < 3).
LCGS_HD void project_backward_pose(const ViewParams& vp, float scale_modifier, float px, float py, float pz, float s0,
                                   float s1, float s2, float qr, float qx, float qy, float qz, const float* g2, float* dpos,
                                   float* dscale, float* drot, float* dview)
{
    project_backward_t<true>(vp, scale_modifier, px, py, pz, s0, s1, s2, qr, qx, qy, qz, g2, dpos, dscale, drot, dview);
}

// The index into vp.view [16] of pose term j < 12 (dview[j] of project_backward_pose).
LCGS_HD int pose_view_index(int j) { return (j / 3) * 4 + j % 3; }

}  // namespace lcgs_b200
