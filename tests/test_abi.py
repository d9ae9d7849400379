"""CPU checks of the boundary: the library builds, loads, and exports what the header declares.

No compute entry point is called here (there is no GPU on the CPU box); argument checks
that return before touching the device are exercised.
"""

import ctypes
import pathlib
import re
import subprocess

import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
HEADER = ROOT / "include" / "momlevel_b200.h"


def _declared():
    text = re.sub(r"/\*.*?\*/", "", HEADER.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(ml_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_path():
    names = _declared()
    for need in ("ml_eos_eval", "ml_flament_spice", "ml_calc_dz", "ml_reference_state", "ml_steric_local",
                 "ml_steric_global", "ml_steric_local_host", "ml_last_error", "ml_version"):
        assert need in names


def test_library_exports_every_declared_symbol():
    from momlevel_b200 import _build, _lib

    path = _build.build()
    assert path.exists()
    out = subprocess.run(["nm", "-D", "--defined-only", str(path)], capture_output=True, text=True, check=True).stdout
    exported = set(re.findall(r"\bT (ml_[a-z0-9_]+)\b", out))
    declared = set(_declared())
    assert declared <= exported, f"missing from the .so: {sorted(declared - exported)}"
    assert set(_lib.EXPORTS) == declared, "ctypes table and header disagree"
    lib = _lib.lib()
    assert lib.ml_version() == 1


def test_library_is_sm100a_only():
    from momlevel_b200 import _build

    out = subprocess.run(["cuobjdump", "-lelf", str(_build.build())], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_(\d+a?)", out))
    assert archs == {"100a"}, archs


def test_argument_errors_are_reported_without_a_device():
    from momlevel_b200 import _lib

    L = _lib.lib()
    # unknown EOS id
    rc = L.ml_eos_eval(7, 0, 0, None, None, 0, 0, None, 0, 1, 1, 1, None, None)
    assert rc == -4 and b"equation of state" in L.ml_last_error()
    # bad dtype
    assert L.ml_flament_spice(5, None, None, 4, None, None) == -3
    # NULL field pointer
    assert L.ml_flament_spice(0, None, None, 4, None, None) == -1
    # empty input is a no-op success (no launch)
    before = L.ml_launch_count()
    assert L.ml_flament_spice(0, None, None, 0, None, None) == 0
    assert L.ml_launch_count() == before
    # both operands broadcast makes no sense
    buf = (ctypes.c_double * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    assert L.ml_eos_eval(0, 0, 1, p, p, 1, 1, p, 0, 1, 1, 1, p, None) == -5
    # misaligned fp64 pointer
    off = ctypes.c_void_p(p.value + 4)
    assert L.ml_eos_eval(0, 0, 1, off, p, 0, 0, p, 0, 1, 1, 1, p, None) == -7
    # workspace too small
    assert L.ml_reference_state(0, 1, p, p, p, p, 1, 1, p, p, p, 8, None) == -6
    with pytest.raises(_lib.MLError):
        _lib.check(-6)


def test_fill_mode_is_checked_before_any_launch():
    """fill_mode is 0 (surface level of every slab) or k in [1, nouter] (every level of slabs [0, k))."""
    from momlevel_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_double * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    before = L.ml_launch_count()
    for fill in (-1, 4):  # nouter = 3
        assert L.ml_adjust_negative_n2(p, fill, 3, 4, 5, p, None) == -5
        assert b"fill_mode" in L.ml_last_error()
        assert L.ml_wave_speed(p, p, fill, 3, 4, 5, p, None) == -5
        assert L.ml_calc_n2(0, 1, p, p, p, -9.8, 101325.0, 1, fill, 3, 4, 5, p, None) == -5
    assert L.ml_launch_count() == before


def test_calc_masso_takes_more_than_65535_rows():
    """More rows than one grid.y are launched in chunks: 65536 rows now reach the workspace check (8 bytes are far
    too few) instead of a shape error; a negative row count is still a shape error.  Neither launches anything."""
    from momlevel_b200 import _lib

    L = _lib.lib()
    buf = (ctypes.c_double * 8)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    before = L.ml_launch_count()
    for dtype in (0, 1):
        assert L.ml_calc_masso(dtype, p, 1, p, 65536, 4, p, p, 8, None) == -6
        assert b"workspace" in L.ml_last_error()
        assert L.ml_calc_masso(dtype, p, 0, None, 70001, 1, p, p, 70001 * 8 - 8, None) == -6
        assert L.ml_calc_masso(dtype, p, 1, p, -1, 4, p, p, 8, None) == -2
    assert L.ml_launch_count() == before


def test_no_product_import_of_the_oracle():
    """The product must never route through the oracle (test infrastructure only)."""
    for path in (ROOT / "momlevel_b200").rglob("*.py"):
        text = path.read_text()
        assert not re.search(r"^\s*(from|import)\s+oracle\b", text, flags=re.M), path
    for path in (ROOT / "momlevel_b200" / "csrc").glob("*"):
        assert "oracle" not in path.read_text(), path
