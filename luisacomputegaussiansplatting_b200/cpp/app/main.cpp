// lcgs-app -- headless CLI of the B200 forward splat renderer.
//
// Keeps the reference CLI's flags and observable behaviour (app/main.cpp:35-343):
//   --res <W>x<H> (default 1600x1063)   --ply <path> (relative paths resolve against argv[0]'s directory)
//   --backend <name> (accepted; always CUDA here, but it still names the output file)
//   --out <dir> (default "out")         --world colmap|blender      --exp_N <frames>      --help / -h
// Output: <out>/<plyname>_<backend>.png, CHW -> HWC with vertical flip and truncating *255
// (main.cpp:322-339) -- in the fused path that conversion is the blend kernel's epilogue, so 3 bytes per
// pixel cross PCIe instead of 12.  The camera pose is the reference's hard-coded one (main.cpp:191-202).
// Extensions: --dump <dir> writes the frame's raw buffers, --fused 0 drives the three reference
// entry points separately instead of the fused frame call, --capacity sets the instance list size L,
// --aux 1 also renders the per-pixel alpha / depth / contributor-count planes (written by --dump).
// --display (ImGui viewer) is out of scope and rejected.
#include <chrono>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <functional>
#include <map>
#include <string>
#include <vector>

#include "gaussians.h"
#include "lcgs/gs_projector.h"
#include "lcgs/gs_tile_splatter.h"
#include "lcgs/sh_preprocessor.h"
#include "lcgs/util/buffer_filler.h"
#include "lcgs/util/camera.h"
#include "lcpp/parallel_primitive.h"
#include "png_writer.h"

namespace fs = std::filesystem;

namespace
{

// Same grammar as the reference's parse_command (app/command_parser.hpp:5-79): any number of leading
// '-', "key=value" or "key value" (the next argument is consumed unless it looks like a flag; a
// leading '-' followed by a digit counts as a value), unknown keys are reported and ignored.
using Handlers = std::map<std::string, std::function<void(const std::string&)>>;

bool parse_command(const Handlers& cmds, int argc, char** argv)
{
    bool ok = true;
    for (int i = 1; i < argc; ++i) {
        const std::string arg = argv[i];
        const size_t      b   = arg.find_first_not_of('-');
        if (b == std::string::npos || b == 0) {
            std::fprintf(stderr, "[lcgs-app] ignoring argument '%s'\n", arg.c_str());
            ok = false;
            continue;
        }
        std::string  key = arg.substr(b), value;
        const size_t eq  = key.find('=');
        if (eq != std::string::npos) {
            value = key.substr(eq + 1);
            key.resize(eq);
        } else if (i + 1 < argc) {
            const std::string next = argv[i + 1];
            const bool flag = !next.empty() && next[0] == '-' && !(next.size() >= 2 && next[1] >= '0' && next[1] <= '9');
            if (!flag) {
                value = next;
                ++i;
            }
        }
        const auto it = cmds.find(key);
        if (it == cmds.end()) {
            std::fprintf(stderr, "[lcgs-app] unknown option '%s'\n", key.c_str());
            ok = false;
        } else {
            it->second(value);
        }
    }
    return ok;
}

template <typename T>
void dump(const fs::path& dir, const char* name, lcgs::Stream& stream, lcgs::BufferView<T> v, size_t n)
{
    std::vector<T> h(n);
    stream.download(v.subview(0, n), h.data());
    stream.synchronize();
    std::ofstream f(dir / name, std::ios::binary);
    f.write(reinterpret_cast<const char*>(h.data()), (std::streamsize)(n * sizeof(T)));
}

}  // namespace

int main(int argc, char** argv)
{
    unsigned    res_w = 1600, res_h = 1063;
    fs::path    ply_path = "gsplat.ply";
    std::string backend = "dx", out_dir = "out", world = "colmap", dump_dir;
    int         exp_N = 1, fused = 1, aux = 0;
    long        capacity = 20000000;  // max num rendered (main.cpp:245)

    Handlers cmds;
    auto     help = [&](const std::string&) {
        std::printf("Usage: %s [options]\n"
                    "  --help / -h              Show this help message\n"
                    "  --res <width>x<height>   Set the resolution (default: %ux%u)\n"
                    "  --ply <path>             Set the path to the PLY file (default: gsplat.ply)\n"
                    "  --backend <name>         Accepted for compatibility (always CUDA sm_100a; default: %s)\n"
                    "  --out <dir>              Set the output directory (default: %s)\n"
                    "  --world <type>           colmap or blender (default: colmap)\n"
                    "  --exp_N <N>              Number of frames to render (default: %d)\n"
                    "  --capacity <L>           Instance list capacity (default: %ld)\n"
                    "  --fused <0|1>            1: fused frame call, 0: SHProcessor/GSProjector/GSTileSplatter (default 1)\n"
                    "  --dump <dir>             Write raw frame buffers for inspection\n"
                    "  --aux <0|1>              1: also render per-pixel alpha, depth and contributor count\n"
                    "                           (alpha.f32, depth_map.f32, n_contrib.u32 under --dump; default 0)\n",
                    argv[0], res_w, res_h, backend.c_str(), out_dir.c_str(), exp_N, capacity);
        std::exit(0);
    };
    cmds["help"] = help;
    cmds["h"]    = help;
    cmds["res"]  = [&](const std::string& s) {
        const size_t x = s.find('x');
        if (x == std::string::npos) lcgs::fatal("Invalid resolution format: '" + s + "'. Expected <width>x<height>");
        res_w = (unsigned)std::stoi(s.substr(0, x));
        res_h = (unsigned)std::stoi(s.substr(x + 1));
    };
    cmds["ply"] = [&](const std::string& s) {
        fs::path p{ s };
        ply_path = p.is_relative() ? fs::path{ argv[0] }.parent_path() / p : p;
    };
    cmds["backend"] = [&](const std::string& s) { backend = s; };
    cmds["out"]     = [&](const std::string& s) { out_dir = s; };
    cmds["world"]   = [&](const std::string& s) {
        if (s.empty() || s == "colmap") world = "colmap";
        else if (s == "blender") world = "blender";
        else lcgs::fatal("Invalid world type: " + s);
    };
    cmds["exp_N"] = [&](const std::string& s) {
        if (s.empty()) lcgs::fatal("--exp_N requires a value");
        exp_N = std::stoi(s);
    };
    cmds["display"]  = [&](const std::string&) { lcgs::fatal("--display (interactive viewer) is not part of this build"); };
    cmds["capacity"] = [&](const std::string& s) { capacity = std::stol(s); };
    cmds["fused"]    = [&](const std::string& s) { fused = s.empty() ? 1 : std::stoi(s); };
    cmds["dump"]     = [&](const std::string& s) { dump_dir = s; };
    cmds["aux"]      = [&](const std::string& s) { aux = s.empty() ? 1 : std::stoi(s); };
    parse_command(cmds, argc, argv);
    if (aux && dump_dir.empty()) {
        std::fprintf(stderr, "[lcgs-app] --aux 1 needs --dump <dir>: the aux planes are only written there\n");
        return 2;
    }

    std::string ply_name = ply_path.filename().string();
    {
        const size_t dot = ply_name.find_last_of('.');
        if (dot == std::string::npos) lcgs::fatal("Invalid ply name: " + ply_name);
        ply_name.resize(dot);
    }
    std::error_code ec;
    fs::create_directories(out_dir, ec);
    if (ec) lcgs::fatal("Failed to create output directory: " + ec.message());
    std::printf("Rendering %s with backend %s, assuming world type %s\n", ply_path.string().c_str(), backend.c_str(),
                world.c_str());

    lcgs::Device device(0);
    lcgs::Stream stream;

    lcgs::GaussiansData data;
    std::string         err;
    if (!lcgs::read_gs_ply(data, ply_path, &err)) lcgs::fatal(err);
    const int P = data.num_gaussians;
    std::printf("num_gaussians: %d\n", P);

    lcgs::GSProjector projector;
    projector.create(device);
    lcgs::BufferFiller                           bf;
    luisa::parallel_primitive::DeviceScan<>      device_scan;
    luisa::parallel_primitive::DeviceRadixSort<> device_radix_sort;
    device_scan.create(device, &stream);
    device_radix_sort.create(device, &stream);
    lcgs::SHProcessor sh_processor;
    sh_processor.create(device);

    auto d_pos     = device.create_buffer<float>((size_t)P * 3);
    auto d_scale   = device.create_buffer<float>((size_t)P * 3);
    auto d_rotq    = device.create_buffer<float>((size_t)P * 4);
    auto d_sh      = device.create_buffer<float>((size_t)P * 16 * 3);
    auto d_color   = device.create_buffer<float>((size_t)P * 3);
    auto d_opacity = device.create_buffer<float>((size_t)P);

    // the reference's hard-coded pose
    lcgs::float3 pos      = { -3.0f, -0.5f, 3.3f };
    lcgs::float3 target   = { 0.0f, 3.0f, 0.5f };
    lcgs::float3 world_up = { 0.0f, -1.0f, -1.0f };
    if (world == "blender") world_up = { 0.0f, 0.0f, 1.0f };
    lcgs::Camera cam = lcgs::get_lookat_cam(pos, target, world_up);
    cam.aspect_ratio = (float)res_w / (float)res_h;
    cam.width        = (int)res_w;
    cam.height       = (int)res_h;
    const lcgs::float3 bg_color = lcgs::make_float3(0.f);

    stream.upload(d_pos.view(), data.pos.data());
    stream.upload(d_scale.view(), data.scale.data());
    stream.upload(d_rotq.view(), data.rotq.data());
    stream.upload(d_sh.view(), data.feature.data());
    stream.upload(d_opacity.view(), data.opacity.data());
    stream.synchronize();

    const auto t_start = std::chrono::steady_clock::now();  // the reference starts its clock here (main.cpp:225-226)
    lcgs::GSTileSplatter tile_splatter;
    tile_splatter.create(device);
    tile_splatter.set_buffer_filler(&bf);
    tile_splatter.set_device_scan(&device_scan);
    tile_splatter.set_device_radix_sort(&device_radix_sort);
    const int  w = (int)res_w, h = (int)res_h;
    const auto tw = (w + tile_splatter.m_blocks.x - 1u) / tile_splatter.m_blocks.x;
    const auto th = (h + tile_splatter.m_blocks.y - 1u) / tile_splatter.m_blocks.y;
    const size_t L = (size_t)capacity;

    auto d_means_2d       = device.create_buffer<float>((size_t)P * 2);
    auto d_depth_features = device.create_buffer<float>((size_t)P);
    auto d_covs_2d        = device.create_buffer<float>((size_t)P * 3);
    auto d_tiles_touched  = device.create_buffer<lcgs::uint>((size_t)P);
    auto d_points_offset  = device.create_buffer<lcgs::uint>((size_t)P);
    auto d_keys_unsorted  = device.create_buffer<lcgs::ulong>(L);
    auto d_list_unsorted  = device.create_buffer<lcgs::uint>(L);
    auto d_keys           = device.create_buffer<lcgs::ulong>(L);
    auto d_list           = device.create_buffer<lcgs::uint>(L);
    auto d_ranges         = device.create_buffer<lcgs::uint>((size_t)tw * th * 2);
    auto d_img            = device.create_buffer<float>((size_t)w * h * 3);
    auto d_radii          = device.create_buffer<int>((size_t)P);
    auto d_alpha          = device.create_buffer<float>(aux ? (size_t)w * h : 1);
    auto d_depth_map      = device.create_buffer<float>(aux ? (size_t)w * h : 1);
    auto d_n_contrib      = device.create_buffer<lcgs::uint>(aux ? (size_t)w * h : 1);
    device.check(lcgs_b200_ctx_reserve(device.ctx(), P, L), "reserve");

    lcgs::GSSplatForwardOutputProxy output{ h, w, d_img, d_radii };
    if (aux) {
        output.target_alpha     = d_alpha.view();
        output.target_depth     = d_depth_map.view();
        output.target_n_contrib = d_n_contrib.view();
    }
    lcgs::GSTileSplatterAccelProxy  accel{ d_tiles_touched, d_points_offset, d_keys_unsorted, d_list_unsorted,
                                          d_keys,          d_list,          d_ranges };
    lcgs::GSTileSplatterInputProxy  input{ P, bg_color, d_means_2d, d_depth_features, d_covs_2d, d_color, d_opacity };

    // fused path: per-scene alpha-test constants (a function of the opacities only) and the uint8 output image
    auto d_alpha_consts = device.create_buffer<float>(fused ? (size_t)P * 2 : 1);
    auto d_rgb8         = device.create_buffer<uint8_t>(fused ? (size_t)w * h * 3 : 1);
    lcgs_b200_scene scene{ P, 3, d_pos.view().ptr, d_scale.view().ptr, d_rotq.view().ptr, d_sh.view().ptr,
                           d_opacity.view().ptr, 1.0f, nullptr };
    if (fused) {
        device.check(lcgs_b200_scene_prepare(device.ctx(), P, d_opacity.view().ptr, d_alpha_consts.view().ptr, stream.abi()),
                     "lcgs_b200_scene_prepare");
        scene.alpha_consts = d_alpha_consts.view().ptr;
    }
    lcgs_b200_frame frame{};
    frame.width = w; frame.height = h;
    frame.means_2d = d_means_2d.view().ptr; frame.depth = d_depth_features.view().ptr; frame.conic = d_covs_2d.view().ptr;
    frame.color = d_color.view().ptr;
    frame.tiles_touched = d_tiles_touched.view().ptr; frame.point_offsets = d_points_offset.view().ptr;
    frame.point_list_keys_unsorted = d_keys_unsorted.view().ptr; frame.point_list_unsorted = d_list_unsorted.view().ptr;
    frame.point_list_keys = d_keys.view().ptr; frame.point_list = d_list.view().ptr;
    frame.ranges = d_ranges.view().ptr; frame.list_capacity = L;
    frame.target_img = d_img.view().ptr; frame.radii = d_radii.view().ptr;
    frame.tile_row_begin = 0; frame.tile_row_end = -1;
    frame.target_rgb8 = fused ? d_rgb8.view().ptr : nullptr;
    if (aux) {
        frame.target_alpha     = d_alpha.view().ptr;
        frame.target_depth     = d_depth_map.view().ptr;
        frame.target_n_contrib = d_n_contrib.view().ptr;
    }

    lcgs::CommandList cmd_list;
    int               num_rendered = 0;
    for (int exp_i = 0; exp_i < exp_N; ++exp_i) {
        if (fused) {
            lcgs_b200_view_params vp;
            lcgs_b200_view_params_from_camera(lcgs::abi(cam), &vp);
            device.check(lcgs_b200_render(device.ctx(), &scene, &vp, &frame, stream.abi()), "lcgs_b200_render");
        } else {
            sh_processor.process(cmd_list, { P, 3, d_pos }, cam, d_sh, d_color, 3, 3);
            projector.forward(cmd_list, { P, d_pos, d_scale, d_rotq, 1.0f }, { d_means_2d, d_covs_2d, d_depth_features }, cam);
            stream << cmd_list.commit();  // main.cpp:270
            num_rendered = tile_splatter.forward(device, stream, accel, input, output);
        }
    }
    if (fused && exp_N > 0) {
        const int rc = lcgs_b200_num_rendered(device.ctx(), stream.abi(), &num_rendered);
        if (rc == LCGS_B200_ERR_CAPACITY) lcgs::fatal(lcgs_b200_last_error(device.ctx()));
        device.check(rc, "lcgs_b200_num_rendered");
    }

    std::vector<float>   h_img(fused ? 0 : (size_t)w * h * 3);
    std::vector<uint8_t> rgb((size_t)w * h * 3);
    std::vector<int>     h_radii((size_t)P);
    if (fused) stream.download(d_rgb8.view(), rgb.data());  // already HWC / flipped / uint8
    else stream.download(d_img.view(), h_img.data());
    stream.download(d_radii.view(), h_radii.data());
    stream.synchronize();
    const double exp_time = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_start).count();
    std::printf("num_rendered: %d\n", num_rendered);
    std::printf("exp time: %f ms\n", exp_time);
    std::printf("fps: %f with test N %d\n", 1000.0 / (exp_time / (exp_N > 0 ? exp_N : 1)), exp_N);

    // 3 x H x W -> H x W x 3, vertical flip, truncating *255 (main.cpp:322-337)
    const size_t plane = (size_t)w * h;
    if (!fused)
        for (int i = 0; i < h; i++)
            for (int j = 0; j < w; j++) {
                const size_t px  = ((size_t)i * w + j) * 3;
                const size_t idx = (size_t)(h - i - 1) * w + j;
                for (int c = 0; c < 3; c++) rgb[px + c] = (uint8_t)(h_img[c * plane + idx] * 255);
            }
    const std::string img_name = out_dir + "/" + ply_name + "_" + backend + ".png";
    if (!lcgs::write_png_rgb8(img_name, w, h, rgb.data())) lcgs::fatal("cannot write " + img_name);
    std::printf("result saved in %s\n", img_name.c_str());

    if (!dump_dir.empty()) {
        fs::create_directories(dump_dir, ec);
        const fs::path d{ dump_dir };
        const size_t   n = (size_t)(num_rendered > 0 ? num_rendered : 0);
        dump(d, "img.f32", stream, d_img.view(), (size_t)w * h * 3);
        dump(d, "radii.i32", stream, d_radii.view(), (size_t)P);
        dump(d, "tiles_touched.u32", stream, d_tiles_touched.view(), (size_t)P);
        dump(d, "depth.f32", stream, d_depth_features.view(), (size_t)P);
        dump(d, "keys_sorted.u64", stream, d_keys.view(), n);
        dump(d, "vals_sorted.u32", stream, d_list.view(), n);
        dump(d, "ranges.u32", stream, d_ranges.view(), (size_t)tw * th * 2);
        if (aux) {
            dump(d, "alpha.f32", stream, d_alpha.view(), (size_t)w * h);
            dump(d, "depth_map.f32", stream, d_depth_map.view(), (size_t)w * h);
            dump(d, "n_contrib.u32", stream, d_n_contrib.view(), (size_t)w * h);
        }
        std::ofstream meta(d / "meta.txt");
        meta << "P " << P << "\nW " << w << "\nH " << h << "\nnum_rendered " << num_rendered << "\n";
    }
    return 0;
}
