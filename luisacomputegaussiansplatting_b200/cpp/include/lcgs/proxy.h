// lcgs/proxy.h -- argument bundles of the splatter, as in the reference's lcgs/include/lcgs/proxy.h:44-73
// (the three structs it declares but never uses, proxy.h:14-42, are omitted).
#pragma once

#include "lcgs/runtime.h"

namespace lcgs
{

struct GSTileSplatterInputProxy {
    int    num_gaussians;
    float3 bg_color;
    BufferView<float> means_2d;        // 2 * P
    BufferView<float> depth_features;  // P
    BufferView<float> conic;           // 3 * P
    BufferView<float> color_features;    // 3 * P
    BufferView<float> opacity_features;  // P
};

struct GSTileSplatterAccelProxy {
    BufferView<uint>  tiles_touched;             // P
    BufferView<uint>  point_offsets;             // P
    BufferView<ulong> point_list_keys_unsorted;  // L
    BufferView<uint>  point_list_unsorted;       // L
    BufferView<ulong> point_list_keys;           // L
    BufferView<uint>  point_list;                // L
    BufferView<uint>  ranges;                    // TW x TH x 2
};

struct GSSplatForwardOutputProxy {
    int               height;
    int               width;
    BufferView<float> target_img;  // planar CHW
    BufferView<int>   radii;       // P
    // extension, optional (empty = off): per-pixel [H][W] planes, see lcgs_b200_frame::target_alpha
    BufferView<float> target_alpha;      // 1 - T
    BufferView<float> target_depth;      // sum of w_i * depth_i (not normalised)
    BufferView<uint>  target_n_contrib;  // Gaussians blended into the pixel
};

}  // namespace lcgs
