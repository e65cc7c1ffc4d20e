"""The C-ABI library builds, loads and exports every symbol include/tip.h declares (no compute calls)."""
import ctypes
import glob
import os
import re

import pytest

from trigenicinteractionpredictor_b200 import _cabi, build


@pytest.fixture(scope="module")
def lib():
    build.build()
    return _cabi.load()


def test_header_and_binding_agree(lib):
    declared = _cabi.header_functions()
    assert declared, "no functions parsed from include/tip.h"
    assert sorted(_cabi.SIGNATURES) == declared
    for name in declared:
        assert hasattr(lib, name), name


def test_trivial_host_only_calls(lib):
    assert lib.tip_abi_version() == 1
    assert lib.tip_stats_len(6000, 10) == 6000 * 10 + 2000 + 1
    assert lib.tip_rows_capacity(1000) >= 2 * 1000 + 62
    assert lib.tip_loglik_workspace_bytes(100, 10) > 0
    assert lib.tip_loglik_workspace_bytes(100, 20) >= lib.tip_loglik_workspace_bytes(100, 10) + 2 * 100 * 400 * 8
    nb = ctypes.c_size_t(0)
    assert lib.tip_em_workspace_bytes(100, 10, 3200, 0, ctypes.byref(nb)) == 0 and nb.value == 2 * 100 * 100 * 8
    assert lib.tip_em_workspace_bytes(100, 4, 3200, 0, ctypes.byref(nb)) == 0 and nb.value == 0
    assert lib.tip_em_workspace_bytes(100, 16, 3200, 0, ctypes.byref(nb)) == 0 and nb.value == 2 * 100 * 256 * 8
    assert lib.tip_em_workspace_bytes(100, 20, 3200, 0, ctypes.byref(nb)) == 0 and nb.value == 4 * 100 * 400 * 8
    assert lib.tip_em_workspace_bytes(100, 20, 3200, 1, ctypes.byref(nb)) == 0 and nb.value == 3200 * 8
    assert lib.tip_em_workspace_bytes(100, 33, 3200, 0, ctypes.byref(nb)) != 0
    assert b"bad arguments" in lib.tip_last_error()


def test_rows_compact_host_format(lib):
    """8-byte host rows: pure host packing (no CUDA call); c | b<<20 | a<<40 | rating<<60 | count<<61."""
    import numpy as np
    rng = np.random.default_rng(3)
    n = 257
    rows = np.empty((n, 4), dtype=np.int32)
    rows[:, :3] = rng.integers(0, 1 << 20, size=(n, 3))
    cnt, rat = rng.integers(0, 8, size=n), rng.integers(0, 2, size=n)
    rows[:, 3] = (cnt << 1) | rat
    out = np.zeros(n, dtype=np.uint64)
    assert lib.tip_rows_compact_host(rows.ctypes.data, n, out.ctypes.data) == 0
    m = np.uint64((1 << 20) - 1)
    assert np.array_equal(out & m, rows[:, 2].astype(np.uint64))
    assert np.array_equal((out >> np.uint64(20)) & m, rows[:, 1].astype(np.uint64))
    assert np.array_equal((out >> np.uint64(40)) & m, rows[:, 0].astype(np.uint64))
    assert np.array_equal((out >> np.uint64(60)) & np.uint64(1), rat.astype(np.uint64))
    assert np.array_equal(out >> np.uint64(61), cnt.astype(np.uint64))
    rows[5, 3] = (8 << 1) | 1                                     # count 8 does not fit
    assert lib.tip_rows_compact_host(rows.ctypes.data, n, out.ctypes.data) != 0
    assert b"row 5" in lib.tip_last_error()
    rows[5, 3] = 2
    rows[7, 1] = 1 << 20                                          # gene id needs 21 bits
    assert lib.tip_rows_compact_host(rows.ctypes.data, n, out.ctypes.data) != 0
    assert lib.tip_rows_compact_host(None, 0, None) == 0


def test_sass_is_sm100a_with_fp64_fma_and_cp_async():
    import shutil
    import subprocess
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("cuobjdump not available")
    out = subprocess.run([cuobjdump, "-sass", _cabi.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out
    assert "DFMA" in out and "LDGSTS" in out and "REDG.E.ADD.F64" in out
    # round 2: the slot-segmented passes run their K^2 work on the fp64 tensor path and are chained by programmatic
    # dependent launches (griddepcontrol.wait = ACQBULK, launch_dependents = PREEXIT); the counting sort ranks with MATCH
    assert "DMMA.8x8x4" in out and "ACQBULK" in out and "PREEXIT" in out and "MATCH.ANY" in out
    # the hot E-step templates are instantiated only for the configurations their launchers select
    assert len(re.findall(r"Function : \S*em_fused_kernel", out)) == 74
    assert len(re.findall(r"Function : \S*seg3_pass_kernel", out)) == 128


def test_environment_reads_are_only_the_kept_hooks():
    """The library and the package read no environment switch beyond the stream-entry hooks: TIP_HOST_NO_STREAM and
    TIP_HOST_SEG3_AFTER_STREAM pick a variant of tip_em_iterations_host, TIP_STREAM_TIMEOUT_US and
    TIP_STREAM_INJECT_FAULT exercise its give-up and checksum-repair paths."""
    pkg = os.path.dirname(os.path.abspath(build.__file__))
    names = set()
    for path in glob.glob(os.path.join(pkg, "csrc", "*.cu")) + glob.glob(os.path.join(pkg, "csrc", "*.cuh")):
        for args in re.findall(r"getenv\(([^)]*)\)", open(path).read()):
            names.update(re.findall(r'"([^"]*)"', args))
    py_read = re.compile(r"""os\.(?:environ\.get|getenv)\(\s*["'](TIP_\w+)["']|os\.environ\[\s*["'](TIP_\w+)["']\s*\](?!\s*=[^=])"""
                         r"""|["'](TIP_\w+)["']\s+(?:not\s+)?in\s+os\.environ""")
    for path in glob.glob(os.path.join(pkg, "**", "*.py"), recursive=True):
        for groups in py_read.findall(open(path).read()):
            names.update(g for g in groups if g)
    assert names == {"TIP_HOST_NO_STREAM", "TIP_HOST_SEG3_AFTER_STREAM", "TIP_STREAM_TIMEOUT_US", "TIP_STREAM_INJECT_FAULT"}
