"""Static checks on the SASS of the shipped library (cuobjdump; no GPU needed): the hot kernels are what DESIGN.md says
they are -- sm_100a only, packed FP32 and asynchronous staging in the blend, no local-memory spills in the production
geometries, no tensor-core or TMA instructions (no stage is a contraction; TMA staging was measured slower)."""
import shutil

import pytest

from luisacomputegaussiansplatting_b200 import build
from sass_ops import kernel_ops

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not available")


@pytest.fixture(scope="module")
def kernels():
    return kernel_ops(build.build_native())


def find(funcs, part):
    hits = [(k, v) for k, v in funcs.items() if part in k]
    assert len(hits) == 1, (part, [k for k, _ in hits])
    return hits[0][1]


def test_library_is_sm_100a_only(kernels):
    archs, funcs = kernels
    assert archs == {"sm_100a"}
    assert len(funcs) >= 20


def test_production_blend_kernel_uses_packed_fp32_and_async_staging(kernels):
    ops = find(kernels[1], "blend2_kernel<10>")
    assert ops["FFMA2"] >= 6 and ops["FMUL2"] >= 4 and ops["FADD2"] >= 2  # the pair's arithmetic of the hit loop
    assert ops["LDGSTS"] >= 3                                             # three 16-byte planes per candidate
    assert ops["MUFU"] >= 2 and ops["FLO"] >= 1 and ops["BMSK"] >= 1
    assert ops["STL"] == 0 and ops["LDL"] == 0
    # the one-pixel-per-lane kernel is not part of the production library
    assert not [k for k in kernels[1] if "blend_kernel<" in k]


def test_production_sort_and_emission_geometries_do_not_spill(kernels):
    funcs = kernels[1]
    for part in ("onesweep_pass_kernel<unsigned long long, 256, 20, 7, 2, false, true>",
                 "onesweep_pass_kernel<unsigned int, 512, 16, 9, 1, false, false>",
                 "duplicate_keys_sorted_kernel<true, true>", "preprocess_fused_kernel<true>", "scan_compact_kernel"):
        ops = find(funcs, part)
        assert ops["STL"] == 0 and ops["LDL"] == 0, part
    assert find(funcs, "onesweep_pass_kernel<unsigned long long, 256, 20, 7, 2, false, true>")["MATCH"] == 0  # ballots
    assert find(funcs, "preprocess_fused_kernel<true>")["LDGSTS"] >= 12                                      # SH rows
    assert find(funcs, "preprocess_fused_kernel<true>")["DFMA"] == 0   # the binary64 threshold sequence left the frame


def test_no_tensor_core_or_tma_instructions(kernels):
    for name, ops in kernels[1].items():
        for op in ("UTCMMA", "HMMA", "UBLKCP", "UTMALDG"):
            assert ops[op] == 0, (name, op)
