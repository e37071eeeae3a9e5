"""The C-ABI library loads and exports exactly the symbols include/gsx.h declares (no compute calls: CPU only)."""
import ctypes
import os
import re

from gradslam_b200 import _C

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared():
    text = open(os.path.join(ROOT, "include", "gsx.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return set(re.findall(r"\b(gsx_[a-z0-9_]+)\s*\(", text))


def test_header_and_binding_list_the_same_symbols():
    assert _declared() == set(_C.SIGNATURES)


def test_library_exports_every_declared_symbol():
    assert os.path.exists(_C.LIB_PATH), "libgsx.so was not built"
    handle = ctypes.CDLL(_C.LIB_PATH)
    for name in sorted(_declared()):
        assert hasattr(handle, name), name


def test_host_only_entry_points():
    lib = _C.lib()
    assert lib.gsx_version() == 201
    n = lib.gsx_fusion_workspace_bytes(8, 480, 640)
    assert n >= 8 * 480 * 640 * 16
    assert 0 < lib.gsx_fusion_workspace_stats_offset(8, 480, 640) < n
    # argument validation happens before any launch, so it is testable without a GPU
    rc = lib.gsx_backproject_normals_fwd(None, 0, None, 0, None, 0, 1, 1, 4, 4, None, None, None, None, None)
    assert rc != 0 and b"null" in lib.gsx_last_error()


def test_no_oracle_import_in_product_package():
    """The product never routes through the oracle (or any CPU fallback)."""
    pkg = os.path.join(ROOT, "gradslam_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "gsx_oracle" not in src and "import oracle" not in src, os.path.join(dirpath, f)


def test_peer_entry_points_check_their_arguments_without_a_gpu():
    """gsx_peer_*: argument validation happens before any CUDA call, so it is testable here."""
    import ctypes

    from gradslam_b200 import _C

    lib = _C.lib()
    buf = (ctypes.c_ubyte * 64)()
    off = ctypes.c_int64(0)
    assert lib.gsx_peer_export(None, buf, ctypes.byref(off), None) != 0
    assert b"gsx_peer_export" in lib.gsx_last_error()
    out = ctypes.c_void_p()
    assert lib.gsx_peer_open(None, 0, ctypes.byref(out)) != 0
    assert lib.gsx_peer_open(buf, -1, ctypes.byref(out)) != 0
    # a block wider than a pitch would overlap the next block
    assert lib.gsx_peer_copy_rows(ctypes.c_void_p(16), 32, ctypes.c_void_p(16), 64, 48, 2, None) != 0
    assert b"gsx_peer_copy_rows" in lib.gsx_last_error()
    # nothing to move is not an error (and touches no pointer)
    assert lib.gsx_peer_copy_rows(None, 32, None, 32, 0, 4, None) == 0
    assert lib.gsx_peer_close_all() == 0
