"""What the built library's hot kernels look like in SASS (cuobjdump on the in-tree .so, no GPU needed).

These are the code-generation facts round 2's measurements rest on (profiles/r2_ab_log.txt): a compiler or
source change that silently undoes one of them costs 5-15 % of a kernel and no parity test would notice.
"""
import re
import shutil
import subprocess

import pytest

from stereoreconstruction_b200 import capi

pytestmark = pytest.mark.skipif(shutil.which("cuobjdump") is None, reason="cuobjdump not on PATH")

BUILD = "_ZN2sr17build_refr_kernelILb1ELb0EEEvNS_13BuildRefrArgsE"
GEO = "_ZN2sr23weights_geodesic_kernelILb1ELi2EEEvNS_10WeightArgsE"
SCREEN = "_ZN2sr24match_mvs_screen2_kernelILi2ELb0ELi2048EEEvNS_9MatchArgsE"


@pytest.fixture(scope="module")
def lib():
    if capi.needs_build():
        capi.build()
    return capi.LIB_PATH


def sass(lib, fun):
    out = subprocess.run(["cuobjdump", "-sass", "-fun", fun, lib], capture_output=True, text=True).stdout
    ops = []
    for line in out.splitlines():
        m = re.match(r"\s+/\*[0-9a-f]{4,5}\*/\s+(.*?);", line)
        if m:
            ops.append(m.group(1).strip())
    assert len(ops) > 100, f"{fun}: not found in {lib}"
    return ops


def resources(lib):
    out = subprocess.run(["cuobjdump", "-res-usage", lib], capture_output=True, text=True).stdout
    res, fun = {}, None
    for line in out.splitlines():
        m = re.search(r"Function (\S+):", line)
        if m:
            fun = m.group(1)
        m = re.search(r"REG:(\d+) STACK:(\d+) SHARED:(\d+)", line)
        if m and fun:
            res[fun] = tuple(int(v) for v in m.groups())
    return res


def test_fp64_clamps_are_compare_select(lib):
    """max.f64 / min.f64 expand to DSETP.MAX/MIN + FSEL + SEL + a NaN fix-up (7 instructions); the build kernel's
    clamps and the geodesic sweeps' minima are setp + selp in PTX (sr_build_refr.cuh clamp_sel, sr_kernels.cuh min_sel)."""
    for fun in (BUILD, GEO):
        bad = [o for o in sass(lib, fun) if re.search(r"DSETP\.(MAX|MIN)", o)]
        assert not bad, f"{fun}: {len(bad)} FP64 min/max expansions, e.g. {bad[0]}"


def test_build_kernel_has_no_conversion_pipe_on_the_label_path(lib):
    """Truncation goes through the 1.5 * 2^52 constant (F2I.F64 issues at 16 lanes/clk/SM; cvt.rzi on the anchor
    labels alone measured 3 % slower)."""
    ops = sass(lib, BUILD)
    assert not [o for o in ops if o.startswith("F2I") and "F64" in o]
    assert sum(1 for o in ops if o.startswith(("DFMA", "DADD", "DMUL"))) > 300


def test_screen_kernel_shape(lib):
    ops = sass(lib, SCREEN)
    ffma2 = sum(1 for o in ops if "FFMA2" in o)
    assert ffma2 >= 50, f"label-vectorised window arithmetic missing ({ffma2} FFMA2)"
    assert not [o for o in ops if "UBLKCP" in o], "bulk async copies (TMA) in the screen: window loads are plain LDG through L1"
    regs, stack, _ = resources(lib)[SCREEN]
    assert regs <= 128, "4 blocks of 128 threads per SM need <= 128 registers"
    assert stack <= 128, f"stack frame grew to {stack} B: spills in the label loop (112 B shipped)"


def test_geodesic_sweeps_are_unrolled_within_six_blocks(lib):
    regs, stack, _ = resources(lib)[GEO]
    assert regs <= 80 and stack == 0, (regs, stack)
