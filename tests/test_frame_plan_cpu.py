"""The fused frame's plan (csrc/frame_plan.cuh), compiled with g++ from tests/frame_plan: over a sweep of scene sizes,
list capacities, tile grids and sort geometries, every region the plan places lies inside what reserve_all reserves,
regions are aligned and disjoint, everything that must start at zero is covered by the frame's one clear kernel, and
neither the tickets nor the clear touch the scalar words that carry results."""
import ctypes as C
import os
import shutil
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "frame_plan", "frame_plan.cpp")
CUDA_INCLUDE = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "include")
SPACE_BITS = 40  # frame_plan.cpp: region space w starts at w << 40
SCAN, SORT, EMIT, SCALARS, RANGES = 1, 2, 3, 4, 5


class Region(C.Structure):
    _fields_ = [("addr", C.c_uint64), ("bytes", C.c_uint64), ("align", C.c_uint64), ("zeroed", C.c_int)]


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    if shutil.which("g++") is None:
        pytest.skip("no C++ compiler")
    if not os.path.exists(os.path.join(CUDA_INCLUDE, "vector_types.h")):
        pytest.skip("no CUDA headers")
    so = str(tmp_path_factory.mktemp("frame_plan") / "libframe_plan.so")
    subprocess.run(["g++", "-O1", "-std=c++17", "-Wall", "-fPIC", "-shared", "-fvisibility=hidden", "-I", CUDA_INCLUDE, SRC,
                    "-o", so], check=True)
    lib = C.CDLL(so)
    lib.fp_plan.argtypes = [C.c_int, C.c_uint64, C.c_uint64, C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.POINTER(Region),
                            C.POINTER(C.c_int), C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
    lib.fp_plan.restype = C.c_int
    return lib


def ceil_log2(v):
    return max(int(v) - 1, 0).bit_length()


def split(addr):
    return addr >> SPACE_BITS, addr & ((1 << SPACE_BITS) - 1)


def plan(lib, P, L, num_tiles, geom):
    reserved = (C.c_uint64 * 3)()
    regions = (Region * 32)()
    clear = (C.c_uint64 * 16)()
    n, nc = C.c_int(), C.c_int()
    rc = lib.fp_plan(P, L, num_tiles, (C.c_int * 6)(*geom), reserved, regions, C.byref(n), clear, C.byref(nc))
    if rc:
        return None
    return list(reserved), [(r.addr, r.bytes, r.align, r.zeroed) for r in regions[:n.value]], \
        [(clear[2 * k], clear[2 * k + 1]) for k in range(nc.value)]


def result_scalars(lib):
    w = (C.c_int * 6)()
    lib.fp_result_scalars(w)
    return list(w[:5]), w[5]


def covered(lo, hi, intervals):
    """[lo, hi) is inside the union of the (start, end) intervals."""
    for s, e in sorted(intervals):
        if s <= lo < e:
            lo = e
        if lo >= hi:
            return True
    return lo >= hi


# (passes come from the key bits) sweep variants of sort.cu, production and tuning: (tile, radix bits)
DEPTH_GEOMS = [(8192, 9), (4096, 9), (2048, 7)]
TILE_GEOMS = [(5120, 7), (4096, 9), (3072, 7), (5376, 7), (6144, 7)]
# (tiles per row, tile rows of the band): one tile, 1080p, 1080p band, 8K, 8K band of one row, 640000 x 48 pixels, the
# widest band and a 65536 x 65536-pixel frame
GRIDS = [(1, 1), (120, 68), (120, 17), (480, 270), (480, 1), (40000, 3), (65535, 1), (4096, 4096)]
SIZES = [(0, 0), (1, 0), (0, 1), (1, 1), (2047, 5000), (2048, 2048), (2049, 100000), (8193, 1 << 16),
         (3_700_000, 17_800_000), (4_000_000, 1_000), (16_000_000, (1 << 30) - 1)]


def test_frame_plan_regions(lib):
    fixed, num_scalars = result_scalars(lib)
    checked = refused = 0
    for P, L in SIZES:
        for gx, rows in GRIDS:
            num_tiles = gx * rows
            bits = ceil_log2(max(num_tiles, 1))
            for dt, dr in DEPTH_GEOMS:
                for tt, tr in TILE_GEOMS:
                    geom = [(32 + dr - 1) // dr, dr, dt, (bits + tr - 1) // tr, tr, tt]
                    got = plan(lib, P, L, num_tiles, geom)
                    if geom[0] > 4 or geom[3] > 4:  # four tickets per sort
                        assert got is None, (P, L, num_tiles, geom)
                        refused += 1
                        continue
                    assert got is not None, ("does not fit what reserve_all reserves", P, L, num_tiles, geom)
                    reserved, regions, clear = got
                    extent = {SCAN: reserved[0], SORT: reserved[1], EMIT: reserved[2], SCALARS: 4 * num_scalars,
                              RANGES: 8 * num_tiles}
                    ctx = (P, L, num_tiles, geom)
                    regions += [((SCALARS << SPACE_BITS) + 4 * w, 4, 4, 0) for w in fixed]
                    for addr, nbytes, align, _ in regions:
                        space, off = split(addr)
                        assert off % align == 0, ctx
                        assert off + nbytes <= extent[space], ("outside the reservation", ctx, space, off, nbytes)
                    spans = sorted((a, a + b) for a, b, _, _ in regions)
                    for (_, e0), (s1, _) in zip(spans, spans[1:]):
                        assert e0 <= s1, ("overlapping regions", ctx)
                    assert len(clear) <= 8, ctx
                    ivs = [(a, a + b) for a, b in clear]
                    for a, b in ivs:
                        space, off = split(a)
                        assert off + (b - a) <= extent[space], ("clear outside the reservation", ctx)
                    for addr, nbytes, _, zeroed in regions:
                        if zeroed:
                            assert covered(addr, addr + nbytes, ivs), ("not cleared", ctx, split(addr), nbytes)
                    for w in fixed:
                        a = (SCALARS << SPACE_BITS) + 4 * w
                        assert not any(s < a + 4 and a < e for s, e in ivs), ("result scalar cleared", ctx, w)
                    checked += 1
    assert checked > 500 and refused > 0
