// Host build of the backward's derivative header (csrc/lcgs_grad.cuh) for tests/test_backward_cpu.py: the same source
// the CUDA kernels inline, compiled with g++ and called through ctypes.  Test-only code.
#include "../../luisacomputegaussiansplatting_b200/csrc/lcgs_grad.cuh"

using namespace lcgs_b200;

#define GM_API extern "C" __attribute__((visibility("default")))

struct ShIn {
    const float* p;
    float operator()(int k, int c) const { return p[k * 3 + c]; }
};
struct ShOut {
    float* p;
    void operator()(int k, int c, float v) const { p[k * 3 + c] = v; }
};

// per Gaussian: g2 [P][12] (packed 2D gradient) -> pos / scale / rotq / sh / opacity gradients, as
// preprocess_backward_kernel computes them for a Gaussian with tiles_touched > 0
GM_API void gm_preprocess_backward(int P, int deg, const float* pos, const float* scale, const float* rotq, const float* sh,
                                   const float* opacity, float scale_modifier, const ViewParams* vp, const float* g2,
                                   float* grad_pos, float* grad_scale, float* grad_rotq, float* grad_sh, float* grad_opacity)
{
    const int feat = (deg + 1) * (deg + 1);
    for (int i = 0; i < P; i++) {
        const float* g = g2 + (size_t)i * kGrad2DFloats;
        float dpos[3] = { 0.f, 0.f, 0.f };
        const float* q = rotq + 4 * (size_t)i;
        project_backward(*vp, scale_modifier, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], scale[3 * i], scale[3 * i + 1],
                         scale[3 * i + 2], q[0], q[1], q[2], q[3], g, dpos, grad_scale + 3 * (size_t)i, grad_rotq + 4 * (size_t)i);
        sh_color_backward(deg, vp->cam_pos, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], ShIn{ sh + (size_t)i * feat * 3 },
                          g + kG2Red, ShOut{ grad_sh + (size_t)i * feat * 3 }, dpos);
        for (int k = 0; k < 3; k++) grad_pos[3 * i + k] = dpos[k];
        grad_opacity[i] = opacity[i] > 0.0f ? g[kG2LogOp] / opacity[i] : 0.0f;
    }
}

// one pixel's walk over n entries: e[n][7] = (dx, dy, a, b, c, ok, alpha_raw), rgb[n][3]; C, G = the pixel's final
// colour and dL/dC.  g[n][9] = per-entry contributions, blended[n] = whether the forward blended the entry.
GM_API void gm_blend_pixel(int n, const float* e, const float* rgb, const float* C, const float* G, float* g, int* blended)
{
    PixelGrad px = pixel_grad_init(true, C, G);
    for (int i = 0; i < n; i++) {
        const float* r = e + 7 * (size_t)i;
        float*       gi = g + (size_t)kGrad2DValues * i;
        for (int k = 0; k < kGrad2DValues; k++) gi[k] = 0.0f;
        blended[i] = blend_entry_grad(px, r[5] != 0.0f, r[6], r[0], r[1], r[2], r[3], r[4], rgb + 3 * (size_t)i, gi) ? 1 : 0;
    }
}
