// Host build of the camera-pose derivatives of csrc/lcgs_grad.cuh (project_backward_pose and the view-direction term
// of sh_color_backward) for tests/test_backward_pose_cpu.py and tests/test_backward_pose.py, compiled with g++ and
// called through ctypes.  Test-only code.
#include "../../luisacomputegaussiansplatting_b200/csrc/lcgs_grad.cuh"

using namespace lcgs_b200;

#define GM_API extern "C" __attribute__((visibility("default")))

struct ShIn {
    const float* p;
    float operator()(int k, int c) const { return p[k * 3 + c]; }
};
struct ShDrop {
    void operator()(int, int, float) const {}
};

// per Gaussian: g2 [P][12] (packed 2D gradient, slot kG2Depth included) -> terms [P][15], the 15 pose terms
// preprocess_pose_grad_kernel sums for a Gaussian with tiles_touched > 0: terms[j] for vp.view[pose_view_index(j)]
// (j < 12) and dL/dcam_pos (j = 12..14)
GM_API void gm_pose_terms(int P, int deg, const float* pos, const float* scale, const float* rotq, const float* sh,
                          float scale_modifier, const ViewParams* vp, const float* g2, float* terms)
{
    const int feat = (deg + 1) * (deg + 1);
    for (int i = 0; i < P; i++) {
        const float* g = g2 + (size_t)i * kGrad2DFloats;
        float*       t = terms + (size_t)i * 15;
        for (int k = 0; k < 15; k++) t[k] = 0.0f;
        float dpos[3] = { 0.f, 0.f, 0.f }, dscale[3], drot[4];
        const float* q = rotq + 4 * (size_t)i;
        project_backward_pose(*vp, scale_modifier, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], scale[3 * i],
                              scale[3 * i + 1], scale[3 * i + 2], q[0], q[1], q[2], q[3], g, dpos, dscale, drot, t);
        float ddir[3] = { 0.f, 0.f, 0.f };
        sh_color_backward(deg, vp->cam_pos, pos[3 * i], pos[3 * i + 1], pos[3 * i + 2], ShIn{ sh + (size_t)i * feat * 3 },
                          g + kG2Red, ShDrop{}, ddir);
        for (int k = 0; k < 3; k++) t[12 + k] = -ddir[k];
    }
}

// The view index of pose term j, as the kernels map it.
GM_API int gm_pose_view_index(int j) { return pose_view_index(j); }
