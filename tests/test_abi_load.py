"""The C-ABI shared library loads and exports every symbol include/hichap_b200.h declares
(no compute calls here: this runs without a GPU)."""
import ctypes
import os
import re

from conftest import ROOT


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "hichap_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(hc_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from hichap_master_b200 import _abi
    assert os.path.isfile(_abi.LIB_PATH), "build first: python -c 'import __graft_entry__ as g; g.build()'"
    handle = ctypes.CDLL(_abi.LIB_PATH)
    syms = declared_symbols()
    assert len(syms) >= 10
    for s in syms:
        assert hasattr(handle, s), "missing export %s" % s


def test_bindings_cover_the_header():
    from hichap_master_b200 import _abi
    assert sorted(_abi.SIGNATURES) == declared_symbols()


def test_version_and_error_string_without_gpu():
    from hichap_master_b200 import _abi
    lib = _abi.lib()
    assert lib.hc_version() == 2
    assert isinstance(lib.hc_last_error(), bytes)
    assert lib.hc_launch_count() >= 0


def test_struct_layout_matches_header():
    from hichap_master_b200 import _abi
    assert ctypes.sizeof(_abi.IceParams) == 40
    assert ctypes.sizeof(_abi.IceResult) == 24
    assert ctypes.sizeof(_abi.IceRunInfo) == 32


def test_ice_stream_kernels_do_not_spill():
    """The <4,2,4> ICE stream kernel sits exactly at the 64-register budget of 4 CTAs/SM; a spill
    costs ~20 % of its bandwidth (profiles/README.md), so the build log is checked.  So is the packed
    kernel's, which has 128 registers at most for its 2 CTAs/SM."""
    log = os.path.join(ROOT, "hichap_master_b200", "csrc", "hc_ice.o.ptxas.log")
    if not os.path.isfile(log):
        import pytest
        pytest.skip("no ptxas log (library built elsewhere)")
    text = open(log).read()
    for name in ("ice_dense_stream_kernelILi4ELi2ELi4E",       # int32 tiles, default variant
                 "ice_q8_mma_kernelENS_"):                     # packed encoding (16 x 128-bit loads in flight)
        m = re.search(name + r".*?\n.*?(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads", text, flags=re.S)
        assert m, name + " not found in the ptxas log"
        assert (int(m.group(2)), int(m.group(3))) == (0, 0), m.group(0)[-120:]
