"""Size of a simulator snapshot (`bd_snapshot_layout`, include/batch_drones.h): a 256-byte header, then the planes, each
starting on a 256-byte boundary.  Host computation only; no GPU needed.  Also: malformed arguments and NULL handles
fail cleanly in every snapshot entry point."""
import ctypes as C
import os
import shutil

import pytest

from marl_gym_pybullet_drones_b200 import _native
from marl_gym_pybullet_drones_b200 import build as bd_build

ANGV, CTRL, EPIS = _native.BD_SNAP_ANGV, _native.BD_SNAP_CTRL, _native.BD_SNAP_EPISODES


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_native.LIB_PATH) or not bd_build.up_to_date():
        if shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"):
            pytest.skip("nvcc not available and library not prebuilt")
        bd_build.build()
    return _native.load()


def _al(x):
    return (x + 255) // 256 * 256


def expected_bytes(N, M, A, B, precision, flags):
    real = 8 if precision else 4
    n = N * M
    b = 256 + 4 * _al(n * 4 * real)               # s0..s3
    if flags & ANGV:
        b += _al(n * 4 * real)                    # s4
    if flags & CTRL:
        b += 13 * _al(n * real)                   # 9 PID memory + 4 commanded-rpm planes
    b += B * _al(n * A * 4)                       # ring, one plane per age
    b += _al(N * 4)                               # step counters
    if flags & EPIS:
        b += _al(N * 4)                           # episode returns
    return b


def layout(lib, N, M, A, B, precision, flags):
    out = C.c_int64(-7)
    rc = lib.bd_snapshot_layout(N, M, A, B, precision, flags, C.byref(out))
    return rc, out.value


@pytest.mark.parametrize("N,M,A,B,precision,flags", [
    (65536, 4, 4, 15, 0, EPIS),            # the headline shape
    (131072, 16, 4, 15, 0, EPIS),          # configs[4]'s per-GPU shape
    (1, 1, 1, 15, 0, 0),                   # every plane far below 256 bytes: padding dominates
    (7, 5, 4, 15, 1, ANGV),                # fp64, odd sizes
    (33, 3, 3, 15, 1, CTRL | EPIS),        # PID
    (10, 2, 4, 25, 0, CTRL),               # VEL, ctrl_freq 50
    (100, 1, 1, 1, 0, ANGV | CTRL | EPIS),
    (64, 2, 4, 15, 0, 0),                  # every plane a multiple of 256 bytes: no padding at all
])
def test_layout_matches_formula(lib, N, M, A, B, precision, flags):
    rc, got = layout(lib, N, M, A, B, precision, flags)
    assert rc == 0
    assert got == expected_bytes(N, M, A, B, precision, flags)
    assert got % 256 == 0


def test_headline_size_and_each_optional_plane(lib):
    rc, base = layout(lib, 65536, 4, 4, 15, 0, 0)
    assert rc == 0
    n = 65536 * 4
    assert base == 256 + 64 * n + 15 * 16 * n + 4 * 65536    # 64 B of state + 240 B of ring per drone, 4 B per env
    assert 79e6 < layout(lib, 65536, 4, 4, 15, 0, EPIS)[1] < 81e6
    assert layout(lib, 65536, 4, 4, 15, 0, ANGV)[1] - base == 16 * n
    assert layout(lib, 65536, 4, 4, 15, 1, ANGV)[1] - layout(lib, 65536, 4, 4, 15, 1, 0)[1] == 32 * n
    assert layout(lib, 65536, 4, 4, 15, 0, CTRL)[1] - base == 13 * 4 * n
    assert layout(lib, 65536, 4, 4, 15, 0, EPIS)[1] - base == 4 * 65536
    # padding: with N = 1, M = 1 every plane takes one 256-byte block
    assert layout(lib, 1, 1, 1, 15, 0, ANGV | CTRL | EPIS)[1] == 256 * (1 + 4 + 1 + 13 + 15 + 1 + 1)


@pytest.mark.parametrize("args", [
    (0, 4, 4, 15, 0, 0), (4, 0, 4, 15, 0, 0), (4, 129, 4, 15, 0, 0), (4, 4, 0, 15, 0, 0), (4, 4, 5, 15, 0, 0),
    (4, 4, 4, 0, 0, 0), (4, 4, 4, 15, 2, 0), (4, 4, 4, 15, -1, 0), (4, 4, 4, 15, 0, 8), (4, 4, 4, 15, 0, -1),
])
def test_malformed_arguments_are_refused(lib, args):
    rc, got = layout(lib, *args)
    assert rc == -1 and got == 0
    assert b"bd_snapshot_layout" in lib.bd_last_error()


def test_null_arguments_fail_cleanly(lib):
    assert lib.bd_snapshot_layout(4, 4, 4, 15, 0, 0, None) == -1
    assert lib.bd_snapshot_bytes(None) == -1
    assert lib.bd_save_snapshot(None, None, None) == -1
    assert b"bd_save_snapshot" in lib.bd_last_error()
    assert lib.bd_load_snapshot(None, None, None, None) == -1
    assert b"bd_load_snapshot" in lib.bd_last_error()
