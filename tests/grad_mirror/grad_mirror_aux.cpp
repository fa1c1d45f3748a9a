// Host build of the aux per-entry step of csrc/lcgs_grad.cuh (pixel_grad_aux_init / blend_entry_grad_aux) for
// tests/test_backward_aux_cpu.py, compiled with g++ and called through ctypes.  Test-only code.
#include "../../luisacomputegaussiansplatting_b200/csrc/lcgs_grad.cuh"

using namespace lcgs_b200;

#define GM_API extern "C" __attribute__((visibility("default")))

// one pixel's walk over n entries: e[n][7] = (dx, dy, a, b, c, ok, alpha_raw), rgb[n][3], z[n] = view depths; C, G =
// the pixel's final colour and dL/dC, A / D = its alpha and depth planes, GA / GD = dL/dA and dL/dD.
// g[n][10] = per-entry contributions (the 10th is dL/dz), blended[n] = whether the forward blended the entry.
GM_API void gm_blend_pixel_aux(int n, const float* e, const float* rgb, const float* z, const float* C, const float* G,
                               float A, float D, float GA, float GD, float* g, int* blended)
{
    PixelGradAux px = pixel_grad_aux_init(true, C, G, A, D, GA, GD);
    for (int i = 0; i < n; i++) {
        const float* r  = e + 7 * (size_t)i;
        float*       gi = g + (size_t)kGrad2DAuxValues * i;
        for (int k = 0; k < kGrad2DAuxValues; k++) gi[k] = 0.0f;
        blended[i] = blend_entry_grad_aux(px, r[5] != 0.0f, r[6], r[0], r[1], r[2], r[3], r[4], rgb + 3 * (size_t)i, z[i], gi)
                         ? 1
                         : 0;
    }
}
