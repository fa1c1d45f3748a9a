// lcgs/gs_tile_splatter.h -- lcgs::GSTileSplatter (reference: lcgs/include/lcgs/gs_tile_splatter.h:19-106,
// lcgs/src/gs_tile_splatter/impl.cpp:63-180).
#pragma once

#include "lcgs/proxy.h"
#include "lcgs/runtime.h"
#include "lcgs/util/buffer_filler.h"
#include "lcpp/parallel_primitive.h"

namespace lcgs
{

class GSTileSplatter : public GSModule
{
public:
    int num_rendered = 0;

    virtual ~GSTileSplatter() = default;
    virtual void create(Device& device) noexcept { m_device = &device; }

    // Same contract as the reference: runs allocate_tiles -> scan -> copy_with_keys -> sort ->
    // get_ranges -> render, mutates input.means_2d / input.conic in place, writes output.radii and
    // returns num_rendered.  It synchronises the stream once (to return the count); the reference
    // synchronises five times (impl.cpp:100,107,131,144,146).
    virtual int forward(Device& device, Stream& stream, GSTileSplatterAccelProxy accel, GSTileSplatterInputProxy input,
                        GSSplatForwardOutputProxy output, bool use_focal = true) noexcept
    {
        forward_async(device, stream, accel, input, output, use_focal);
        const int rc = lcgs_b200_num_rendered(device.ctx(), stream.abi(), &num_rendered);
        if (rc == LCGS_B200_ERR_CAPACITY) fatal(std::string("GSTileSplatter::forward: ") + lcgs_b200_last_error(device.ctx()));
        device.check(rc, "GSTileSplatter::forward");
        return num_rendered;
    }

    // Extension: enqueue only; fetch the count later with lcgs_b200_num_rendered.
    void forward_async(Device& device, Stream& stream, GSTileSplatterAccelProxy accel, GSTileSplatterInputProxy input,
                       GSSplatForwardOutputProxy output, bool use_focal = true) noexcept
    {
        if (!use_focal) fatal("GSTileSplatter::forward(use_focal=false) is not implemented");
        lcgs_b200_frame f{};
        f.width = output.width; f.height = output.height;
        f.bg_color[0] = input.bg_color.x; f.bg_color[1] = input.bg_color.y; f.bg_color[2] = input.bg_color.z;
        f.means_2d = input.means_2d.ptr; f.depth = input.depth_features.ptr; f.conic = input.conic.ptr;
        f.color = input.color_features.ptr;
        f.tiles_touched = accel.tiles_touched.ptr; f.point_offsets = accel.point_offsets.ptr;
        f.point_list_keys_unsorted = accel.point_list_keys_unsorted.ptr; f.point_list_unsorted = accel.point_list_unsorted.ptr;
        f.point_list_keys = accel.point_list_keys.ptr; f.point_list = accel.point_list.ptr;
        f.ranges = accel.ranges.ptr;
        size_t cap = accel.point_list_keys_unsorted.count;
        if (accel.point_list_unsorted.count < cap) cap = accel.point_list_unsorted.count;
        if (accel.point_list_keys.count < cap) cap = accel.point_list_keys.count;
        if (accel.point_list.count < cap) cap = accel.point_list.count;
        f.list_capacity = cap;
        f.target_img = output.target_img.ptr; f.radii = output.radii.ptr;
        f.target_alpha = output.target_alpha.ptr; f.target_depth = output.target_depth.ptr;
        f.target_n_contrib = output.target_n_contrib.ptr;
        f.tile_row_begin = 0; f.tile_row_end = -1;
        device.check(lcgs_b200_splat_forward(device.ctx(), input.num_gaussians, input.opacity_features.ptr, &f, stream.abi()),
                     "GSTileSplatter::forward");
    }

    // The reference stores raw non-owning pointers to these helpers; scan, sort and fill live inside
    // the lcgs_b200 context here, the setters are kept for source compatibility.
    BufferFiller* mp_buffer_filler = nullptr;
    void          set_buffer_filler(BufferFiller* bf) noexcept { mp_buffer_filler = bf; }
    luisa::parallel_primitive::DeviceScan<>*      mp_device_scan       = nullptr;
    luisa::parallel_primitive::DeviceRadixSort<>* mp_device_radix_sort = nullptr;
    void set_device_scan(luisa::parallel_primitive::DeviceScan<>* scan) noexcept { mp_device_scan = scan; }
    void set_device_radix_sort(luisa::parallel_primitive::DeviceRadixSort<>* sort) noexcept { mp_device_radix_sort = sort; }
};

}  // namespace lcgs
