"""ctypes front-end of tests/oracle_aux/oracle_aux.c (test infrastructure only): the CPU oracle's blend plus the
per-pixel aux planes.  The library is compiled once per process into a temporary directory (never into the tree),
with the oracle's own compiler flags (oracle/Makefile), so its arithmetic is the oracle's."""
from __future__ import annotations

import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "oracle_aux", "oracle_aux.c")
_CFLAGS = ["-O2", "-mavx2", "-mfma", "-ffp-contract=off", "-fno-math-errno", "-fopenmp", "-fPIC", "-fvisibility=hidden"]
_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="lcgs_aux_oracle_")
        atexit.register(shutil.rmtree, d, True)
        so = os.path.join(d, "liboracle_aux.so")
        subprocess.run(["gcc", *_CFLAGS, "-shared", "-o", so, _SRC, "-lm"], check=True)
        _lib = C.CDLL(so)
        _lib.orc_blend_aux.restype = None
    return _lib


def _p(a: np.ndarray):
    return a.ctypes.data_as(C.c_void_p)


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def blend_aux(W, H, bg, ranges, point_list, means_pix, conic, opacity, color, depth, row0: int = 0,
              row1: int = -1) -> dict:
    """K9 plus the aux planes: img [3,H,W], n_examined, alpha = 1 - T, depth_map = sum of w * depth (blend order, not
    normalised) and n_contrib = entries blended, each [H,W].  Rows outside the band stay 0."""
    img = np.zeros((3, H, W), np.float32)
    nex = np.zeros((H, W), np.uint32)
    alpha = np.zeros((H, W), np.float32)
    dmap = np.zeros((H, W), np.float32)
    ncon = np.zeros((H, W), np.uint32)
    lib().orc_blend_aux(C.c_int(W), C.c_int(H), _p(_f32(bg)), _p(np.ascontiguousarray(ranges, np.uint32)),
                        _p(np.ascontiguousarray(point_list, np.uint32)), _p(_f32(means_pix)), _p(_f32(conic)),
                        _p(_f32(opacity)), _p(_f32(color)), _p(img), _p(nex), C.c_int(row0), C.c_int(row1),
                        _p(_f32(depth)), _p(alpha), _p(dmap), _p(ncon))
    return dict(img=img, n_examined=nex, alpha=alpha, depth_map=dmap, n_contrib=ncon)
