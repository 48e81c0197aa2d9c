"""The C-ABI library loads and exports every symbol include/cavb200.h declares, and the ctypes
binding covers exactly that set (no compute calls: this runs without a GPU)."""
import ctypes
import os
import re

from cav_hoomd_b200 import capi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, "include", "cavb200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cavb200_[a-z0-9_]+)\s*\(", text)))


def test_header_declares_the_expected_entry_points():
    syms = header_symbols()
    for must in ("cavb200_create", "cavb200_force", "cavb200_force_read", "cavb200_bussi", "cavb200_bussi_ke",
                 "cavb200_step", "cavb200_step_host", "cavb200_rhok", "cavb200_fkt", "cavb200_shard_step",
                 "cavb200_track_record", "cavb200_track_record_from", "cavb200_track_set_reference_from"):
        assert must in syms


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(capi.LIB_PATH)
    missing = [s for s in header_symbols() if not hasattr(lib, s)]
    assert not missing, missing


def test_ctypes_binding_covers_the_header_exactly():
    assert sorted(capi._SIGNATURES) == header_symbols()


def test_version_and_struct_layouts():
    lib = capi.load()
    assert lib.cavb200_version() == 100
    assert ctypes.sizeof(capi.Params) == 32  # struct cavity_force_params: 4 doubles (reference .h:28-54)
    assert ctypes.sizeof(capi.BussiArgs) == 48
    p = capi.Params.make(0.01, 1e-3, 2.0)
    assert p.K == 2.0 * 0.01 * 0.01


def test_no_cpu_fallback_without_a_device():
    """Without a CUDA device create() fails with a CUDA error; nothing computes on the CPU."""
    import pytest
    if os.path.exists("/dev/nvidiactl"):
        pytest.skip("a GPU is present")
    with pytest.raises(capi.CavbError):
        capi.Handle(0)


def test_product_does_not_import_the_oracle():
    """Nothing under cav_hoomd_b200/ (or the C-ABI sources) may reference oracle/."""
    bad = []
    pkg = os.path.join(ROOT, "cav_hoomd_b200")
    for d, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cc")):
                txt = open(os.path.join(d, f), errors="ignore").read()
                if re.search(r"^\s*(from|import)\s+oracle\b|#include\s+[\"<].*oracle", txt, flags=re.M):
                    bad.append(os.path.join(d, f))
    assert not bad, bad
