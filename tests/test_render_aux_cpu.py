"""Static checks of the per-pixel aux outputs (no GPU needed): the ctypes frame matches the C header's layout, and the
shipped library's aux blend kernel is what DESIGN.md says (sm_100a, no spills, depth staged with cp.async, packed FP32)."""
import ctypes
import os
import shutil
import subprocess

import pytest

from luisacomputegaussiansplatting_b200 import _capi, build
from sass_ops import kernel_ops

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.skipif(shutil.which("cc") is None, reason="no C compiler")
def test_ctypes_frame_matches_the_header(tmp_path):
    fields = [name for name, _ in _capi.Frame._fields_]
    assert fields[-3:] == ["target_alpha", "target_depth", "target_n_contrib"]
    src = tmp_path / "layout.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "lcgs_b200.h"\nint main(void) {\n'
                   '    printf("sizeof %zu\\n", sizeof(lcgs_b200_frame));\n'
                   + "".join('    printf("%s %%zu\\n", offsetof(lcgs_b200_frame, %s));\n' % (f, f) for f in fields)
                   + "    return 0;\n}\n")
    exe = tmp_path / "layout"
    subprocess.run(["cc", "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe)], check=True)
    out = dict(ln.split() for ln in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    assert int(out["sizeof"]) == ctypes.sizeof(_capi.Frame)
    for f in fields:
        assert int(out[f]) == getattr(_capi.Frame, f).offset, f


@pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")
def test_aux_blend_kernel_sass():
    archs, funcs = kernel_ops(build.build_native())
    assert archs == {"sm_100a"}
    hits = [v for k, v in funcs.items() if "blend2_aux_kernel<" in k]
    assert len(hits) == 1, [k for k in funcs if "aux" in k]
    ops = hits[0]
    assert ops["STL"] == 0 and ops["LDL"] == 0
    assert ops["LDGSTS"] >= 4   # three 16-byte record planes + the 4-byte depth per candidate
    assert ops["FFMA2"] >= 7    # the pair's arithmetic plus the depth accumulator


def test_cli_aux_needs_dump(tmp_path):
    r = subprocess.run([build.build_app(), "--aux", "1", "--out", str(tmp_path)], capture_output=True, text=True, timeout=60)
    assert r.returncode == 2 and "--dump" in r.stderr
