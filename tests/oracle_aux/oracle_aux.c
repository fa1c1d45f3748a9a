/* TEST INFRASTRUCTURE ONLY: the CPU oracle's blend with the per-pixel aux planes of lcgs_b200_frame.
 *
 * The oracle itself (oracle/lcgs_oracle.c) is compiled into this library unchanged, so the walk below uses the very same
 * orc_exp / orc_alpha_passes.  orc_blend_aux repeats orc_blend's per-pixel walk (K9, shader.cpp:171-288) statement for
 * statement and adds, in the oracle's non-fused style:
 *   alpha[pix]     = 1 - T
 *   depth_map[pix] = D, D = D + wgt * depth[id] over the blended entries, in blend order (not normalised)
 *   n_contrib[pix] = number of blended entries (entries rejected by power > 0 or the alpha test and the entry that
 *                    saturates the pixel are not counted -- unlike n_examined, the reference's `contributor`)
 * img and n_examined are orc_blend's outputs; tests/test_oracle_aux.py checks them against orc_blend bit for bit.
 * Each of alpha / depth_map / n_contrib (W*H) may be NULL; depth is needed when depth_map is given.  Rows
 * [row0*16, min(H, row1*16)) are written, tile ids are band-local. */
#include "../../oracle/lcgs_oracle.c"

ORC_API void orc_blend_aux(int W, int H, const float* bg, const uint32_t* ranges, const uint32_t* point_list,
                           const float* means_2d, const float* conic, const float* opacity, const float* color,
                           float* img, uint32_t* n_examined, int row0, int row1, const float* depth, float* alpha,
                           float* depth_map, uint32_t* n_contrib)
{
    int gx = (W + 15) / 16, gy = (H + 15) / 16;
    if (row1 < 0) row1 = gy;
    size_t plane = (size_t)W * (size_t)H;
    int    ntile = gx * (row1 - row0);
#pragma omp parallel for schedule(dynamic, 1)
    for (int t = 0; t < ntile; t++) {
        int      bx = t % gx, by = row0 + t / gx;
        uint32_t start = ranges[2 * t], end = ranges[2 * t + 1];
        for (int ly = 0; ly < 16; ly++)
            for (int lx = 0; lx < 16; lx++) {
                int px = bx * 16 + lx, py = by * 16 + ly;
                if (px >= W || py >= H) continue;
                float    pxf = (float)px, pyf = (float)py;
                float    T = 1.0f, C[3] = { 0.0f, 0.0f, 0.0f }, D = 0.0f;
                uint32_t contributor = 0, blended = 0;
                for (uint32_t k = start; k < end; k++) {
                    contributor++;
                    uint32_t id = point_list[k];
                    float dx = means_2d[2 * (size_t)id] - pxf;
                    float dy = means_2d[2 * (size_t)id + 1] - pyf;
                    float cx = conic[3 * (size_t)id], cy = conic[3 * (size_t)id + 1], cz = conic[3 * (size_t)id + 2];
                    float op = opacity[id];
                    float power = fmaf(-(cy * dx), dy, fmaf((-0.5f * cx) * dx, dx, ((-0.5f * cz) * dy) * dy));
                    if (power > 0.0f) continue;
                    float a;
                    if (!orc_alpha_passes(op, power, &a)) continue;
                    float test_T = T * (1.0f - a);
                    if (test_T < 0.0001f) break; /* saturated: this entry is not blended */
                    float wgt = T * a;
                    C[0] = C[0] + wgt * color[3 * (size_t)id];
                    C[1] = C[1] + wgt * color[3 * (size_t)id + 1];
                    C[2] = C[2] + wgt * color[3 * (size_t)id + 2];
                    if (depth_map) D = D + wgt * depth[id];
                    blended++;
                    T = test_T;
                }
                size_t pix = (size_t)px + (size_t)W * (size_t)py;
                for (int c = 0; c < 3; c++) img[pix + c * plane] = bg[c] * T + C[c];
                if (n_examined) n_examined[pix] = contributor;
                if (alpha) alpha[pix] = 1.0f - T;
                if (depth_map) depth_map[pix] = D;
                if (n_contrib) n_contrib[pix] = blended;
            }
    }
}
