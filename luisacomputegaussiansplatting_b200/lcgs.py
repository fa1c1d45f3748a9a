"""Host-side mirror of the reference's `lcgs` library interface over the C ABI.

Same class and method names, argument meaning and side effects as the reference's C++ classes
(SHProcessor, GSProjector, GSTileSplatter, BufferFiller, the proxies, Camera and its helpers), with
torch CUDA tensors standing in for luisa::compute::BufferView<T> and a torch stream for
Stream/CommandList.  PyTorch only provides device memory and streams here; every kernel is ours
(liblcgs_b200.so) and nothing runs without it.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence

import numpy as np
import torch

from . import _capi
from ._capi import Camera, CapacityError, LcgsError, ViewParams  # noqa: F401  (re-exported)


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), "buffers must be contiguous CUDA tensors"
    return t.data_ptr()


def _stream_handle(stream: Optional[torch.cuda.Stream]) -> Optional[int]:
    s = stream if stream is not None else torch.cuda.current_stream()
    return s.cuda_stream or None


# --------------------------------------------------------------------------------------------------
# camera (lcgs/include/lcgs/util/camera.h)
# --------------------------------------------------------------------------------------------------

def get_lookat_cam(pos: Sequence[float], target: Sequence[float], world_up: Sequence[float]) -> Camera:
    """lcgs::get_lookat_cam, camera.h:74-82."""
    cam = Camera()
    _capi.check(_capi.load().lcgs_b200_get_lookat_cam(_capi.fvec(pos), _capi.fvec(target), _capi.fvec(world_up),
                                                      C.byref(cam)))
    return cam


def make_camera(pos, target, world_up, width: int, height: int, fov: float = 60.0) -> Camera:
    """get_lookat_cam followed by the assignments of app/main.cpp:204-207."""
    cam = get_lookat_cam(pos, target, world_up)
    cam.fov = fov
    cam.aspect_ratio = float(np.float32(width) / np.float32(height))
    cam.width = int(width)
    cam.height = int(height)
    return cam


def _mat(fn, *args) -> np.ndarray:
    m = (C.c_float * 16)()
    _capi.check(fn(*args, m))
    return np.array(m, np.float32)


def local_to_world_matrix(cam: Camera) -> np.ndarray:
    return _mat(_capi.load().lcgs_b200_local_to_world_matrix, C.byref(cam))


def world_to_local_matrix(cam: Camera) -> np.ndarray:
    return _mat(_capi.load().lcgs_b200_world_to_local_matrix, C.byref(cam))


def projection_matrix(tanfovx: float, tanfovy: float, znear: float = 0.1, zfar: float = 100.0) -> np.ndarray:
    return _mat(_capi.load().lcgs_b200_projection_matrix, tanfovx, tanfovy, znear, zfar)


def view_params(cam: Camera) -> ViewParams:
    """Host prologue of GSProjector::forward (gs_projector/impl.cpp:34-42)."""
    vp = ViewParams()
    _capi.check(_capi.load().lcgs_b200_view_params_from_camera(C.byref(cam), C.byref(vp)))
    return vp


# --------------------------------------------------------------------------------------------------
# device
# --------------------------------------------------------------------------------------------------

class Device:
    """Stands in for luisa::compute::Device + the module create() calls: owns one lcgs_b200 context."""

    def __init__(self, index: int = 0):
        self.lib = _capi.load()
        if not torch.cuda.is_available():
            raise LcgsError(_capi.ERR_NO_DEVICE, "no CUDA device (there is no CPU fallback)")
        self.index = index
        self.torch_device = torch.device("cuda", index)
        torch.cuda.set_device(index)
        ctx = C.c_void_p()
        _capi.check(self.lib.lcgs_b200_ctx_create(index, C.byref(ctx)))
        self.ctx = ctx

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.lcgs_b200_ctx_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, status: int):
        _capi.check(status, self.ctx)

    def create_buffer(self, dtype: torch.dtype, n: int) -> torch.Tensor:
        """Device::create_buffer<T>(n).  Zero-initialised (the reference's buffers are not)."""
        return torch.zeros(int(n), dtype=dtype, device=self.torch_device)

    def reserve(self, num_gaussians: int, max_instances: int):
        self.check(self.lib.lcgs_b200_ctx_reserve(self.ctx, int(num_gaussians), int(max_instances)))

    def set_profiling(self, on: bool):
        self.check(self.lib.lcgs_b200_set_profiling(self.ctx, 1 if on else 0))

    def stage_times(self) -> dict:
        ms = (C.c_float * _capi.NUM_STAGES)()
        self.check(self.lib.lcgs_b200_stage_times(self.ctx, ms))
        return dict(zip(_capi.STAGES, [float(x) for x in ms]))

    def sort_breakdown(self) -> dict:
        h, p, k = C.c_float(), C.c_float(), C.c_int()
        self.check(self.lib.lcgs_b200_sort_breakdown(self.ctx, C.byref(h), C.byref(p), C.byref(k)))
        return dict(histogram_ms=h.value, passes_ms=p.value, num_passes=k.value)

    # ---- multi-GPU flow control (device-side sequence flags in a peer buffer) and the consumer's checksum ----
    def peer_signal(self, flag_ptr: int, value: int, stream: Optional[torch.cuda.Stream] = None):
        self.check(self.lib.lcgs_b200_peer_signal(self.ctx, C.c_void_p(int(flag_ptr)), int(value) & 0xFFFFFFFF,
                                                  _stream_handle(stream)))

    def peer_wait(self, flag_ptr: int, value: int, timeout_ms: int = 5000, stream: Optional[torch.cuda.Stream] = None):
        self.check(self.lib.lcgs_b200_peer_wait(self.ctx, C.c_void_p(int(flag_ptr)), int(value) & 0xFFFFFFFF, int(timeout_ms),
                                                _stream_handle(stream)))

    def peer_timeouts(self) -> int:
        n = C.c_uint32()
        self.check(self.lib.lcgs_b200_peer_error(self.ctx, C.byref(n)))
        return int(n.value)

    def checksum_u32(self, data_ptr: int, num_words: int, out: torch.Tensor, stream: Optional[torch.cuda.Stream] = None):
        """out: one int64 device element = wrap-around sum of the 32-bit words at data_ptr."""
        self.check(self.lib.lcgs_b200_checksum_u32(self.ctx, C.c_void_p(int(data_ptr)), int(num_words), out.data_ptr(),
                                                   _stream_handle(stream)))

    def num_rendered(self, stream: Optional[torch.cuda.Stream] = None) -> int:
        n = C.c_int()
        self.check(self.lib.lcgs_b200_num_rendered(self.ctx, _stream_handle(stream), C.byref(n)))
        return n.value


# --------------------------------------------------------------------------------------------------
# proxies (lcgs/include/lcgs/proxy.h, gs_projector.h:16-28, sh_preprocessor.h:16-20)
# --------------------------------------------------------------------------------------------------

@dataclass
class GPUPointsProxy:
    N: int
    stride: int
    pos: torch.Tensor


@dataclass
class GSProjectorInputProxy:
    num_gaussians: int
    pos: torch.Tensor
    scale: torch.Tensor
    rotq: torch.Tensor
    scale_modifier: float = 1.0


@dataclass
class GSProjectorOutputProxy:
    means_2d: torch.Tensor
    covs_2d: torch.Tensor
    depth: torch.Tensor


@dataclass
class GSTileSplatterInputProxy:
    num_gaussians: int
    bg_color: Sequence[float]
    means_2d: torch.Tensor
    depth_features: torch.Tensor
    conic: torch.Tensor
    color_features: torch.Tensor
    opacity_features: torch.Tensor


@dataclass
class GSTileSplatterAccelProxy:
    tiles_touched: torch.Tensor
    point_offsets: torch.Tensor
    point_list_keys_unsorted: torch.Tensor
    point_list_unsorted: torch.Tensor
    point_list_keys: torch.Tensor
    point_list: torch.Tensor
    ranges: torch.Tensor


@dataclass
class GSSplatForwardOutputProxy:
    height: int
    width: int
    target_img: torch.Tensor
    radii: torch.Tensor
    # extension, optional: per-pixel [H*W] planes (see Renderer(aux=True)); None = not rendered
    target_alpha: Optional[torch.Tensor] = None       # float32, 1 - T
    target_depth: Optional[torch.Tensor] = None       # float32, sum of w_i * depth_i
    target_n_contrib: Optional[torch.Tensor] = None   # int32 / uint32, Gaussians blended


# --------------------------------------------------------------------------------------------------
# modules
# --------------------------------------------------------------------------------------------------

class SHProcessor:
    """lcgs::SHProcessor (sh_preprocessor.h:22-57)."""

    def create(self, device: Device):
        self.device = device

    def process(self, stream, proxy: GPUPointsProxy, camera: Camera, sh: torch.Tensor, color: torch.Tensor,
                channel: int = 3, level: int = 3):
        """Enqueue only.  As in the reference, the 6th positional argument is what the kernel uses
        as the SH degree (header/implementation swap, SURVEY.md Q9); both are 3 in the app."""
        d = self.device
        deg = channel
        d.check(d.lib.lcgs_b200_sh_process(d.ctx, int(proxy.N), int(deg), _capi.fvec(list(camera.position)),
                                           _ptr(proxy.pos), _ptr(sh), _ptr(color), _stream_handle(stream)))


class GSProjector:
    """lcgs::GSProjector (gs_projector.h:30-87)."""

    m_blocks = (16, 16)

    def create(self, device: Device):
        self.device = device

    def forward(self, stream, input: GSProjectorInputProxy, output: GSProjectorOutputProxy, cam: Camera,
                use_focal: bool = True):
        if not use_focal:
            raise LcgsError(_capi.ERR_UNSUPPORTED, "use_focal=False is unreachable from the app and mis-scales "
                                                   "cov.z upstream (SURVEY.md Q11); not implemented")
        d = self.device
        vp = view_params(cam)
        d.check(d.lib.lcgs_b200_project(d.ctx, int(input.num_gaussians), _ptr(input.pos), _ptr(input.scale),
                                        _ptr(input.rotq), float(input.scale_modifier), C.byref(vp),
                                        _ptr(output.means_2d), _ptr(output.depth), _ptr(output.covs_2d),
                                        _stream_handle(stream)))


class BufferFiller:
    """lcgs::BufferFiller (util/buffer_filler.h)."""

    block_size = 256

    def fill(self, device: Device, buffer_view: torch.Tensor, v, stream=None):
        fn = {torch.int32: device.lib.lcgs_b200_fill_u32, torch.uint32: device.lib.lcgs_b200_fill_u32,
              torch.int64: device.lib.lcgs_b200_fill_u64, torch.uint64: device.lib.lcgs_b200_fill_u64,
              torch.float32: device.lib.lcgs_b200_fill_f32}[buffer_view.dtype]
        device.check(fn(device.ctx, _ptr(buffer_view), buffer_view.numel(), v, _stream_handle(stream)))


class DeviceScan:
    """luisa::parallel_primitive::DeviceScan<> as used at gs_tile_splatter/impl.cpp:34,104."""

    def create(self, device: Device, stream=None):
        self.device, self.stream = device, stream

    @staticmethod
    def GetTempStorageBytes(num_items: int) -> int:
        return int(_capi.load().lcgs_b200_scan_temp_bytes(int(num_items)))

    def InclusiveSum(self, stream, d_in: torch.Tensor, d_out: torch.Tensor, num_items: int):
        d = self.device
        d.check(d.lib.lcgs_b200_scan_inclusive_u32(d.ctx, _ptr(d_in), _ptr(d_out), int(num_items),
                                                   _stream_handle(stream)))


class DeviceRadixSort:
    """luisa::parallel_primitive::DeviceRadixSort<> as used at gs_tile_splatter/impl.cpp:50,135-143."""

    def create(self, device: Device, stream=None):
        self.device, self.stream = device, stream

    @staticmethod
    def GetSortPairsTempStorageBytes(num_items: int) -> int:
        return int(_capi.load().lcgs_b200_sort_temp_bytes(int(num_items)))

    def SortPairs(self, stream, keys_in, keys_out, vals_in, vals_out, num_items: int, begin_bit: int = 0,
                  end_bit: int = 64):
        d = self.device
        d.check(d.lib.lcgs_b200_sort_pairs_u64_u32(d.ctx, _ptr(keys_in), _ptr(keys_out), _ptr(vals_in),
                                                   _ptr(vals_out), int(num_items), int(begin_bit), int(end_bit),
                                                   _stream_handle(stream)))


def _frame_struct(accel: GSTileSplatterAccelProxy, inp: GSTileSplatterInputProxy, out: GSSplatForwardOutputProxy,
                  row_begin: int = 0, row_end: int = -1) -> _capi.Frame:
    f = _capi.Frame()
    f.width, f.height = int(out.width), int(out.height)
    f.bg_color[:] = [float(x) for x in inp.bg_color]
    f.means_2d, f.depth, f.conic, f.color = _ptr(inp.means_2d), _ptr(inp.depth_features), _ptr(inp.conic), _ptr(
        inp.color_features)
    f.tiles_touched, f.point_offsets = _ptr(accel.tiles_touched), _ptr(accel.point_offsets)
    f.point_list_keys_unsorted, f.point_list_unsorted = _ptr(accel.point_list_keys_unsorted), _ptr(
        accel.point_list_unsorted)
    f.point_list_keys, f.point_list = _ptr(accel.point_list_keys), _ptr(accel.point_list)
    f.ranges = _ptr(accel.ranges)
    f.list_capacity = min(accel.point_list_keys_unsorted.numel(), accel.point_list_unsorted.numel(),
                          accel.point_list_keys.numel(), accel.point_list.numel())
    f.target_img, f.radii = _ptr(out.target_img), _ptr(out.radii)
    f.tile_row_begin, f.tile_row_end = int(row_begin), int(row_end)
    f.target_alpha, f.target_depth = _ptr(out.target_alpha), _ptr(out.target_depth)
    f.target_n_contrib = _ptr(out.target_n_contrib)
    return f


class GSTileSplatter:
    """lcgs::GSTileSplatter (gs_tile_splatter.h:19-106)."""

    m_blocks = (16, 16)

    def __init__(self):
        self.num_rendered = 0
        self.mp_buffer_filler = None
        self.mp_device_scan = None
        self.mp_device_radix_sort = None

    def create(self, device: Device):
        self.device = device

    # the reference stores raw non-owning pointers; scan/sort/fill live inside the C-ABI context here
    def set_buffer_filler(self, bf: BufferFiller):
        self.mp_buffer_filler = bf

    def set_device_scan(self, scan: DeviceScan):
        self.mp_device_scan = scan

    def set_device_radix_sort(self, sort: DeviceRadixSort):
        self.mp_device_radix_sort = sort

    def forward_async(self, device: Device, stream, accel: GSTileSplatterAccelProxy, input: GSTileSplatterInputProxy,
                      output: GSSplatForwardOutputProxy, use_focal: bool = True, tile_rows=(0, -1)):
        """Enqueue the whole splat (no host synchronisation at all)."""
        if not use_focal:
            raise LcgsError(_capi.ERR_UNSUPPORTED, "use_focal=False not implemented (SURVEY.md Q11)")
        f = _frame_struct(accel, input, output, *tile_rows)
        device.check(device.lib.lcgs_b200_splat_forward(device.ctx, int(input.num_gaussians),
                                                        _ptr(input.opacity_features), C.byref(f),
                                                        _stream_handle(stream)))

    def forward(self, device: Device, stream, accel, input, output, use_focal: bool = True, tile_rows=(0, -1)) -> int:
        """GSTileSplatter::forward: returns num_rendered (synchronises once, where the reference does
        five times).  Mutates input.means_2d (-> pixels) and input.conic (-> inverse covariance) and
        writes output.radii, like the reference (Q7)."""
        self.forward_async(device, stream, accel, input, output, use_focal, tile_rows)
        self.num_rendered = device.num_rendered(stream)
        return self.num_rendered


# --------------------------------------------------------------------------------------------------
# fused frame renderer (what the app's loop does, app/main.cpp:266-308)
# --------------------------------------------------------------------------------------------------

def transpose_rgba8(device: Device, img_chw: torch.Tensor, width: int, height: int, out: Optional[torch.Tensor] = None,
                    stream: Optional[torch.cuda.Stream] = None) -> torch.Tensor:
    """Display::_transpose_shader (app/display.cpp:30-39): planar float image -> [H, W, 4] RGBA8 framebuffer."""
    if out is None:
        out = torch.empty((height, width, 4), dtype=torch.uint8, device=img_chw.device)
    device.check(device.lib.lcgs_b200_transpose_rgba8(device.ctx, int(width), int(height), _ptr(img_chw), _ptr(out),
                                                      _stream_handle(stream)))
    return out


class PeerBuffer:
    """Device memory on the `owner` rank that every rank of the process group can write with plain stores
    over NVLink (lcgs_b200_peer_alloc / _open: CUDA IPC + peer access).  Passed as a render target, the
    blend kernel's image stores are the transfer: finished frames / tile-row strips land on the owner
    without a separate collective.  `ptr` is valid in the calling process only."""

    def __init__(self, device: Device, nbytes: int, owner: int = 0, group=None):
        import torch.distributed as dist

        self.device, self.nbytes, self.owner = device, int(nbytes), owner
        self.rank = dist.get_rank(group)
        self.is_owner = self.rank == owner
        p = C.c_void_p()
        handle = C.create_string_buffer(_capi.PEER_HANDLE_BYTES)
        if self.is_owner:
            device.check(device.lib.lcgs_b200_peer_alloc(device.ctx, self.nbytes, C.byref(p), handle))
        box = [handle.raw if self.is_owner else None]
        dist.broadcast_object_list(box, src=owner, group=group)
        if not self.is_owner:
            device.check(device.lib.lcgs_b200_peer_open(device.ctx, box[0], C.byref(p)))
        self.ptr = int(p.value)

    def to_host(self, offset_bytes: int, count: int) -> np.ndarray:
        """float32 view of [offset, offset + 4*count) copied to the host (synchronises the device)."""
        out = np.empty(count, dtype=np.float32)
        torch.cuda.synchronize()
        d = self.device
        d.check(d.lib.lcgs_b200_peer_read(d.ctx, C.c_void_p(self.ptr + offset_bytes), out.ctypes.data_as(C.c_void_p), 4 * count))
        return out

    def close(self):
        if self.ptr:
            d = self.device
            torch.cuda.synchronize()
            d.check((d.lib.lcgs_b200_peer_free if self.is_owner else d.lib.lcgs_b200_peer_close)(d.ctx, C.c_void_p(self.ptr)))
            self.ptr = 0


class Renderer:
    """Device-resident scene + frame buffers + the fused lcgs_b200_render call."""

    def __init__(self, device: Device, pos, scale, rotq, sh, opacity, width: int, height: int,
                 list_capacity: int = 20_000_000, sh_deg: int = 3, scale_modifier: float = 1.0,
                 bg_color=(0.0, 0.0, 0.0), tile_rows=(0, -1), keep_intermediates: bool = True,
                 rgb8: bool = False, prepare_scene: bool = True, aux: bool = False):
        """rgb8: the blend kernel also writes the app's uint8 HWC image (main.cpp:322-337) into `self.rgb8`.
        aux: the blend kernel also writes three per-pixel planes -- accumulated opacity (`alpha()`), the sum of
        weight * view depth over the blended Gaussians (`depth_map()`, see `expected_depth()`) and the number of
        Gaussians blended into the pixel (`n_contrib()`).
        prepare_scene: compute the per-scene alpha-test constants once (lcgs_b200_scene_prepare) instead of
        deriving them from the opacity in every frame; call `scene_changed()` after modifying `opacity`."""
        self.device = device
        dev = device.torch_device

        def up(a, dt=torch.float32):
            t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(a))
            return t.to(device=dev, dtype=dt).contiguous()

        # main.cpp:180-223: five arrays uploaded once
        self.pos, self.scale, self.rotq, self.sh, self.opacity = up(pos), up(scale), up(rotq), up(sh), up(opacity)
        P = self.P = int(self.pos.shape[0])
        self.W, self.H = int(width), int(height)
        self.gx, self.gy = (self.W + 15) // 16, (self.H + 15) // 16
        r0, r1 = tile_rows
        r1 = self.gy if r1 < 0 else r1
        self.tile_rows = (r0, r1)
        self.num_tiles = self.gx * (r1 - r0)
        self.capacity = int(list_capacity)
        z = lambda n, dt: torch.zeros(int(n), dtype=dt, device=dev)  # noqa: E731
        # main.cpp:232-254: the 12 frame buffers
        self.means_2d = z(2 * P, torch.float32) if keep_intermediates else None
        self.depth = z(P, torch.float32)
        self.conic = z(3 * P, torch.float32) if keep_intermediates else None
        self.color = z(3 * P, torch.float32) if keep_intermediates else None
        self.tiles_touched = z(P, torch.int32)
        self.point_offsets = z(P, torch.int32)
        self.keys_unsorted = z(self.capacity, torch.int64)
        self.vals_unsorted = z(self.capacity, torch.int32)
        self.keys = z(self.capacity, torch.int64)
        self.vals = z(self.capacity, torch.int32)
        self.ranges = z(2 * max(self.gx * self.gy, 1), torch.int32)  # sized for the whole frame: bands can be re-cut
        self.img = z(3 * self.W * self.H, torch.float32)
        self.radii = z(P, torch.int32)
        self.rgb8 = torch.zeros(3 * self.W * self.H, dtype=torch.uint8, device=dev) if rgb8 else None
        self.alpha_consts = z(2 * P, torch.float32) if prepare_scene else None
        # per-pixel planes ([H*W]; `self.depth` is the per-Gaussian depth)
        self.alpha_map = z(self.W * self.H, torch.float32) if aux else None
        self.depth_plane = z(self.W * self.H, torch.float32) if aux else None
        self.n_contrib_map = z(self.W * self.H, torch.int32) if aux else None

        self.c_scene = _capi.Scene(P, int(sh_deg), _ptr(self.pos), _ptr(self.scale), _ptr(self.rotq), _ptr(self.sh),
                                   _ptr(self.opacity), float(scale_modifier), _ptr(self.alpha_consts))
        f = self.c_frame = _capi.Frame()
        f.width, f.height = self.W, self.H
        f.bg_color[:] = [float(x) for x in bg_color]
        f.means_2d, f.depth, f.conic, f.color = _ptr(self.means_2d), _ptr(self.depth), _ptr(self.conic), _ptr(
            self.color)
        f.tiles_touched, f.point_offsets = _ptr(self.tiles_touched), _ptr(self.point_offsets)
        f.point_list_keys_unsorted, f.point_list_unsorted = _ptr(self.keys_unsorted), _ptr(self.vals_unsorted)
        f.point_list_keys, f.point_list = _ptr(self.keys), _ptr(self.vals)
        f.ranges, f.list_capacity = _ptr(self.ranges), self.capacity
        f.target_img, f.radii = _ptr(self.img), _ptr(self.radii)
        f.tile_row_begin, f.tile_row_end = r0, r1
        f.target_rgb8 = _ptr(self.rgb8)
        f.target_alpha, f.target_depth = _ptr(self.alpha_map), _ptr(self.depth_plane)
        f.target_n_contrib = _ptr(self.n_contrib_map)
        device.reserve(P, self.capacity)
        self.scene_changed()

    def set_tile_rows(self, r0: int, r1: int):
        """Render tile rows [r0, r1) from the next frame on (tile-row sharding: bands re-balanced between frames)."""
        assert 0 <= r0 <= r1 <= self.gy
        self.tile_rows = (r0, r1)
        self.num_tiles = self.gx * (r1 - r0)
        self.c_frame.tile_row_begin, self.c_frame.tile_row_end = r0, r1

    def scene_changed(self, stream: Optional[torch.cuda.Stream] = None):
        """Refresh the per-scene constants derived from `opacity` (no-op without prepare_scene)."""
        if self.alpha_consts is not None:
            d = self.device
            d.check(d.lib.lcgs_b200_scene_prepare(d.ctx, self.P, _ptr(self.opacity), _ptr(self.alpha_consts),
                                                  _stream_handle(stream)))

    def nbytes_scene(self) -> int:
        return sum(t.numel() * t.element_size() for t in (self.pos, self.scale, self.rotq, self.sh, self.opacity))

    def render_async(self, vp: ViewParams, stream: Optional[torch.cuda.Stream] = None):
        d = self.device
        d.check(d.lib.lcgs_b200_render(d.ctx, C.byref(self.c_scene), C.byref(vp), C.byref(self.c_frame),
                                       _stream_handle(stream)))

    def render(self, cam: Camera, stream: Optional[torch.cuda.Stream] = None) -> int:
        """One frame; returns num_rendered (raises CapacityError if it exceeds list_capacity)."""
        self.render_async(view_params(cam), stream)
        return self.device.num_rendered(stream)

    def read_image(self, host_img: torch.Tensor, stream: Optional[torch.cuda.Stream] = None):
        """main.cpp:313-315: enqueue the D2H copy of the planar image into pinned host memory."""
        d = self.device
        d.check(d.lib.lcgs_b200_read_image(d.ctx, C.byref(self.c_frame), host_img.data_ptr(), _stream_handle(stream)))

    def read_image_rgb8(self, host_rgb: torch.Tensor, stream: Optional[torch.cuda.Stream] = None):
        """Enqueue the D2H copy of the fused uint8 HWC image (3*W*H bytes) into pinned host memory."""
        d = self.device
        d.check(d.lib.lcgs_b200_read_image_rgb8(d.ctx, C.byref(self.c_frame), host_rgb.data_ptr(), _stream_handle(stream)))

    def set_target_rgb8(self, rgb: Optional[torch.Tensor]):
        assert rgb is None or (rgb.numel() == 3 * self.W * self.H and rgb.dtype == torch.uint8)
        self.rgb8 = rgb
        self.c_frame.target_rgb8 = _ptr(rgb)

    def set_target(self, img: torch.Tensor):
        """Render the following frames into another planar [3*H*W] float32 device buffer."""
        assert img.numel() == 3 * self.W * self.H and img.dtype == torch.float32
        self.img = img
        self.c_frame.target_img = _ptr(img)

    def set_target_ptr(self, ptr: int, rgb8_ptr: Optional[int] = None):
        """Render the following frames into raw device memory (e.g. a slot of a PeerBuffer on another GPU):
        a planar [3*H*W] float32 image at `ptr` (and, optionally, the uint8 HWC image at `rgb8_ptr`).
        `image()` keeps referring to the local buffer."""
        self.c_frame.target_img = C.c_void_p(int(ptr))
        if rgb8_ptr is not None:
            self.c_frame.target_rgb8 = C.c_void_p(int(rgb8_ptr)) if rgb8_ptr else None

    def read_num_rendered_async(self, host_count: torch.Tensor, stream: Optional[torch.cuda.Stream] = None):
        """Enqueue a copy of the last enqueued frame's num_rendered into a pinned int32 host tensor."""
        d = self.device
        d.check(d.lib.lcgs_b200_read_num_rendered_async(d.ctx, host_count.data_ptr(), _stream_handle(stream)))

    def image(self) -> torch.Tensor:
        return self.img.view(3, self.H, self.W)

    def _aux_plane(self, t: Optional[torch.Tensor]) -> torch.Tensor:
        if t is None:
            raise LcgsError(_capi.ERR_INVALID, "the per-pixel planes need Renderer(..., aux=True)")
        return t.view(self.H, self.W)

    def alpha(self) -> torch.Tensor:
        """[H, W] float32: accumulated opacity 1 - T of the last frame (same row order as `image()`)."""
        return self._aux_plane(self.alpha_map)

    def depth_map(self) -> torch.Tensor:
        """[H, W] float32: sum over the blended Gaussians of weight * view depth, in blend order (not normalised)."""
        return self._aux_plane(self.depth_plane)

    def n_contrib(self) -> torch.Tensor:
        """[H, W] int32: number of Gaussians blended into each pixel (the saturating entry is not counted)."""
        return self._aux_plane(self.n_contrib_map)

    def expected_depth(self) -> torch.Tensor:
        """[H, W] float32: depth_map / alpha where alpha > 0, else 0."""
        a, d = self.alpha(), self.depth_map()
        return torch.where(a > 0, d / torch.where(a > 0, a, torch.ones_like(a)), torch.zeros_like(d))

    def intermediates(self, n: Optional[int] = None) -> dict:
        """Host copies of every buffer of the last frame, typed like the oracle's Frame."""
        n = self.device.num_rendered() if n is None else n
        u32 = lambda t: t.cpu().numpy().view(np.uint32)  # noqa: E731
        out = dict(
            num_rendered=n, depth=self.depth.cpu().numpy(),
            tiles_touched=u32(self.tiles_touched), radii=self.radii.cpu().numpy(), offsets=u32(self.point_offsets),
            keys_unsorted=self.keys_unsorted[:n].cpu().numpy().view(np.uint64), vals_unsorted=u32(self.vals_unsorted[:n]),
            keys_sorted=self.keys[:n].cpu().numpy().view(np.uint64), vals_sorted=u32(self.vals[:n]),
            ranges=u32(self.ranges).reshape(-1, 2)[:self.num_tiles], img=self.image().cpu().numpy())
        if self.alpha_map is not None:
            out["alpha"] = self.alpha().cpu().numpy()
            out["depth_map"] = self.depth_map().cpu().numpy()
            out["n_contrib"] = u32(self.n_contrib_map).reshape(self.H, self.W)
        if self.conic is not None:
            out["means_2d"] = self.means_2d.cpu().numpy().reshape(-1, 2)
            out["conic"] = self.conic.cpu().numpy().reshape(-1, 3)
            out["color"] = self.color.cpu().numpy().reshape(-1, 3)
        return out


# --------------------------------------------------------------------------------------------------
# differentiable rendering (extension: no reference counterpart)
# --------------------------------------------------------------------------------------------------

def _scene_input(t: torch.Tensor, device: torch.device) -> torch.Tensor:
    """float32, contiguous, 16-byte aligned copy (or the tensor itself when it already is one), detached."""
    t = t.detach().to(device=device, dtype=torch.float32).contiguous()
    return t if t.data_ptr() % 16 == 0 else t.clone()


class _RenderFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dr: "DifferentiableRenderer", vp: ViewParams, pos, scale, rotq, sh, opacity):
        img, (scene, b) = dr._forward(vp, pos, scale, rotq, sh, opacity)
        # the image is the output: it goes through save_for_backward (an attribute would make a reference cycle)
        ctx.save_for_backward(img)
        ctx.dr, ctx.vp, ctx.saved = dr, vp, (scene, {k: v for k, v in b.items() if k != "img"})
        ctx.shapes = [t.shape for t in (pos, scale, rotq, sh, opacity)]
        return img

    @staticmethod
    def backward(ctx, dl_dimg):
        want = ctx.needs_input_grad[2:]
        scene, b = ctx.saved
        b = dict(b, img=ctx.saved_tensors[0])
        grads = ctx.dr._backward(ctx.vp, (scene, b), dl_dimg, want)
        ctx.saved = None  # the frame's buffers are released with the graph
        out = [g.view(s) if g is not None else None for g, s in zip(grads, ctx.shapes)]
        return (None, None, *out)


class _RenderAuxFunction(torch.autograd.Function):
    """_RenderFunction with the alpha and depth planes as two more outputs.  Gradients are not materialised: a plane
    the loss does not use reaches the C call as NULL (the image-only blend backward then runs), and an unused image
    as a zero gradient."""

    @staticmethod
    def forward(ctx, dr: "DifferentiableRenderer", vp: ViewParams, pos, scale, rotq, sh, opacity):
        img, (scene, b) = dr._forward(vp, pos, scale, rotq, sh, opacity)
        alpha, depth = b["alpha_plane"].view(dr.H, dr.W), b["depth_plane"].view(dr.H, dr.W)
        ctx.set_materialize_grads(False)
        ctx.save_for_backward(img, alpha, depth)
        ctx.dr, ctx.vp = dr, vp
        ctx.saved = (scene, {k: v for k, v in b.items() if k not in ("img", "alpha_plane", "depth_plane")})
        ctx.shapes = [t.shape for t in (pos, scale, rotq, sh, opacity)]
        return img, alpha, depth

    @staticmethod
    def backward(ctx, dl_dimg, dl_dalpha, dl_ddepth):
        want = ctx.needs_input_grad[2:]
        scene, b = ctx.saved
        img, alpha, depth = ctx.saved_tensors
        b = dict(b, img=img, alpha_plane=alpha, depth_plane=depth)
        if dl_dimg is None:
            dl_dimg = torch.zeros_like(img)
        grads = ctx.dr._backward(ctx.vp, (scene, b), dl_dimg, want, dl_dalpha, dl_ddepth)
        ctx.saved = None
        out = [g.view(s) if g is not None else None for g, s in zip(grads, ctx.shapes)]
        return (None, None, *out)


class DifferentiableRenderer:
    """Renders one whole frame as the output of a torch.autograd.Function: `dr(pos, scale, rotq, sh, opacity, cam)`
    returns the planar [3, H, W] image, and `backward` runs lcgs_b200_render_backward (CUDA kernels, no reference
    counterpart) to produce gradients shaped like the five inputs.  The inputs are the scene arrays after activation
    (pos [P,3], scale [P,3], rotq [P,4] = (r,x,y,z), sh [P,(sh_deg+1)^2,3], opacity [P]); chaining to pre-activation
    parameters is ordinary torch code around the call.  The image is bit-identical to `Renderer.render`'s.

    Each call allocates the buffers its backward reads (instance list, ranges, means_2d, conic, colour,
    tiles_touched, image) and keeps them on the autograd graph, so several views may be rendered before one
    `loss.backward()`.  The unsorted / sorted key lists are scratch shared by every call of this renderer.  The
    alpha-test constants are recomputed every call, because the opacity changes every step.  A frame with more
    instances than `list_capacity` raises CapacityError in the forward.

    keep_means_2d_grad: keep the last backward's [P, 2] pixel-space mean gradient (the densification statistic) in
    `means_2d_grad`.

    aux: the call returns `(img [3, H, W], alpha [H, W], depth [H, W])`, the planes of `Renderer(aux=True)`:
    accumulated opacity 1 - T and the sum of weight * view depth over the blended Gaussians (not normalised; the
    expected depth is `depth / alpha` where alpha > 0, ordinary torch code).  All three are differentiable, so mask,
    depth and opacity losses train the scene; the image is bit-identical to the one without aux."""

    def __init__(self, device: Device, width: int, height: int, list_capacity: int = 4_000_000, sh_deg: int = 3,
                 bg_color=(0.0, 0.0, 0.0), scale_modifier: float = 1.0, keep_means_2d_grad: bool = False,
                 aux: bool = False):
        self.device = device
        self.W, self.H = int(width), int(height)
        self.gx, self.gy = (self.W + 15) // 16, (self.H + 15) // 16
        self.capacity = int(list_capacity)
        self.sh_deg = int(sh_deg)
        self.bg_color = tuple(float(x) for x in bg_color)
        self.scale_modifier = float(scale_modifier)
        self.keep_means_2d_grad = keep_means_2d_grad
        self.means_2d_grad: Optional[torch.Tensor] = None
        self.aux = bool(aux)
        dev = device.torch_device
        self.keys_unsorted = torch.zeros(self.capacity, dtype=torch.int64, device=dev)
        self.vals_unsorted = torch.zeros(self.capacity, dtype=torch.int32, device=dev)
        self.keys = torch.zeros(self.capacity, dtype=torch.int64, device=dev)
        self._reserved = -1

    def __call__(self, pos, scale, rotq, sh, opacity, cam: Camera):
        fn = _RenderAuxFunction if self.aux else _RenderFunction
        return fn.apply(self, view_params(cam), pos, scale, rotq, sh, opacity)

    def _scene(self, pos, scale, rotq, sh, opacity, alpha_consts) -> _capi.Scene:
        P = int(pos.shape[0])
        return _capi.Scene(P, self.sh_deg, _ptr(pos), _ptr(scale), _ptr(rotq), _ptr(sh), _ptr(opacity),
                           self.scale_modifier, _ptr(alpha_consts))

    def _frame(self, b: dict) -> _capi.Frame:
        f = _capi.Frame()
        f.width, f.height = self.W, self.H
        f.bg_color[:] = list(self.bg_color)
        f.means_2d, f.depth, f.conic, f.color = _ptr(b["means_2d"]), _ptr(b["depth"]), _ptr(b["conic"]), _ptr(b["color"])
        f.tiles_touched, f.point_offsets = _ptr(b["tiles_touched"]), _ptr(b["point_offsets"])
        f.point_list_keys_unsorted, f.point_list_unsorted = _ptr(self.keys_unsorted), _ptr(self.vals_unsorted)
        f.point_list_keys, f.point_list = _ptr(self.keys), _ptr(b["point_list"])
        f.ranges, f.list_capacity = _ptr(b["ranges"]), self.capacity
        f.target_img, f.radii = _ptr(b["img"]), _ptr(b["radii"])
        f.tile_row_begin, f.tile_row_end = 0, -1
        f.target_alpha, f.target_depth = _ptr(b.get("alpha_plane")), _ptr(b.get("depth_plane"))
        return f

    def _forward(self, vp: ViewParams, pos, scale, rotq, sh, opacity):
        d = self.device
        dev = d.torch_device
        feat = (self.sh_deg + 1) ** 2
        P = int(pos.shape[0])
        assert tuple(sh.shape) == (P, feat, 3), "sh must be [P, (sh_deg+1)^2, 3]"
        assert vp.width == self.W and vp.height == self.H, "camera resolution differs from the renderer's"
        scene = [_scene_input(t, dev) for t in (pos, scale, rotq, sh, opacity)]
        if P > self._reserved:
            d.reserve(P, self.capacity)
            self._reserved = P
        z = lambda n, dt: torch.zeros(int(n), dtype=dt, device=dev)  # noqa: E731
        b = dict(means_2d=z(2 * P, torch.float32), depth=z(P, torch.float32), conic=z(3 * P, torch.float32),
                 color=z(3 * P, torch.float32), tiles_touched=z(P, torch.int32), point_offsets=z(P, torch.int32),
                 point_list=torch.empty(self.capacity, dtype=torch.int32, device=dev),
                 ranges=z(2 * max(self.gx * self.gy, 1), torch.int32), img=z(3 * self.W * self.H, torch.float32),
                 radii=z(P, torch.int32), alpha_consts=torch.empty(2 * P, dtype=torch.float32, device=dev))
        if self.aux:
            b.update(alpha_plane=z(self.W * self.H, torch.float32), depth_plane=z(self.W * self.H, torch.float32))
        stream = _stream_handle(None)
        d.check(d.lib.lcgs_b200_scene_prepare(d.ctx, P, _ptr(scene[4]), _ptr(b["alpha_consts"]), stream))
        c_scene = self._scene(*scene, b["alpha_consts"])
        f = self._frame(b)
        d.check(d.lib.lcgs_b200_render(d.ctx, C.byref(c_scene), C.byref(vp), C.byref(f), stream))
        d.num_rendered()  # raises CapacityError on overflow
        return b["img"].view(3, self.H, self.W), (scene, b)

    def _backward(self, vp: ViewParams, saved, dl_dimg: torch.Tensor, want, dl_dalpha=None, dl_ddepth=None) -> list:
        d = self.device
        scene, b = saved
        P = int(scene[0].shape[0])
        dl = dl_dimg.detach().to(dtype=torch.float32).contiguous()
        planes = [None if t is None else t.detach().to(dtype=torch.float32).contiguous() for t in (dl_dalpha, dl_ddepth)]
        grads = [torch.empty_like(t) if w else None for t, w in zip(scene, want)]
        g = _capi.Grad()
        g.dl_dimg = _ptr(dl)
        g.dl_dalpha, g.dl_ddepth = _ptr(planes[0]), _ptr(planes[1])
        g.grad_pos, g.grad_scale, g.grad_rotq, g.grad_sh, g.grad_opacity = (_ptr(t) for t in grads)
        m2 = torch.empty((P, 2), dtype=torch.float32, device=dl.device) if self.keep_means_2d_grad else None
        g.grad_means_2d = _ptr(m2)
        c_scene = self._scene(*scene, b["alpha_consts"])
        f = self._frame(b)
        d.check(d.lib.lcgs_b200_render_backward(d.ctx, C.byref(c_scene), C.byref(vp), C.byref(f), C.byref(g),
                                                _stream_handle(None)))
        if self.keep_means_2d_grad:
            self.means_2d_grad = m2
        return grads
