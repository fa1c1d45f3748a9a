// Host build of the SSIM loss's per-pixel arithmetic (csrc/ssim_math.cuh) for tests/test_ssim_cpu.py, compiled with
// g++ and called through ctypes.  Test-only code.
#include "../../luisacomputegaussiansplatting_b200/csrc/ssim_math.cuh"

using namespace lcgs_b200;

#define SM_API extern "C" __attribute__((visibility("default")))

// m [5][n] (mx, my, exx, eyy, exy) -> out [4][n] (s, P0, P1, P2)
SM_API void sm_ssim_pixel(int n, const float* m, float* out)
{
    for (int i = 0; i < n; i++) {
        const SsimPixel p = ssim_pixel(m[i], m[n + i], m[2 * n + i], m[3 * n + i], m[4 * n + i]);
        out[i] = p.s;
        out[n + i] = p.p0;
        out[2 * n + i] = p.p1;
        out[3 * n + i] = p.p2;
    }
}

SM_API float sm_ssim_weight(int k) { return ssim_weight(k); }
