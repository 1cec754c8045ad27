"""CPU-side checks of the C-ABI shared library: it builds for sm_100a, loads, and exports every
symbol include/lstep_b200.h declares. No compute calls (no GPU here)."""
import ctypes
import os
import re

from lstep_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "lstep_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(lstep_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_header_symbols():
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    names = declared_symbols()
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"{n} declared in lstep_b200.h but not exported"
    assert set(names) == set(_lib.EXPORTS), set(names) ^ set(_lib.EXPORTS)


def test_status_strings_and_sizes():
    lib = _lib.load(require_device=False)
    assert lib.lstep_abi_version() == 2
    assert lib.lstep_strerror(0) == b"ok"
    assert lib.lstep_packed_ld(172) == 192
    small = lib.lstep_update_pe_workspace_bytes(10, 10, 4, 12, 10, 61)
    big = lib.lstep_update_pe_workspace_bytes(300, 200, 20, 172, 100, 10985)
    assert 0 < small < big
    assert lib.lstep_update_pe_workspace_bytes(-1, 0, 4, 12, 10, 61) == 0
    assert lib.lstep_csr_build_workspace_bytes(1000, 50) > 1000 * 36


def test_sass_is_sm100a_only():
    """The library carries sm_100a code and nothing else (no multi-arch fatbin)."""
    import subprocess
    out = subprocess.run([build.cuobjdump(), "-lelf", build.LIB], capture_output=True, text=True).stdout
    archs = set(re.findall(r"sm_\d+a?", out))
    assert archs == {"sm_100a"}, archs
