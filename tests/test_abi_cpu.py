"""The C-ABI shared library loads without a GPU and exports every symbol include/scannet_b200.h declares.
No compute entry point is called here (they need a B200 and fail loudly without one)."""
import ctypes as C
import os
import re

from scannet_b200._lib import LIB_PATH, lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    src = open(os.path.join(ROOT, "include", "scannet_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(scn_[a-z0-9_]+)\s*\(", src)))


def test_every_declared_symbol_is_exported(built):
    L = lib()
    syms = declared_symbols()
    assert len(syms) >= 40
    missing = [s for s in syms if not hasattr(L, s)]
    assert not missing, missing


def test_library_is_self_contained(built):
    """no torch / oracle dependency in the product library"""
    import subprocess
    out = subprocess.run(["ldd", LIB_PATH], capture_output=True, text=True).stdout
    assert "oracle" not in out and "torch" not in out and "libref" not in out


def test_no_gpu_means_loud_failure_not_fallback(built):
    L = lib()
    n = L.scn_device_count()
    if n > 0:
        return                      # on the GPU box this test has nothing to show
    from scannet_b200 import ScnError, segmentator, tsdf
    import numpy as np
    import pytest
    with pytest.raises(ScnError):
        tsdf.TsdfVolume(tsdf.default_params(max_blocks=16, hash_slots=64))
    with pytest.raises(ScnError):
        segmentator.segment_mesh(np.zeros((3, 3), np.float32), np.array([[0, 1, 2]], np.uint32))


def test_product_never_imports_oracle():
    """oracle/ is test infrastructure: nothing under scannet_b200/ may reference it"""
    bad = []
    for dp, _, fs in os.walk(os.path.join(ROOT, "scannet_b200")):
        for f in fs:
            if f.endswith((".py", ".cu", ".cpp", ".h", ".cuh")):
                txt = open(os.path.join(dp, f), errors="replace").read()
                if re.search(r"(import|include|CDLL|dlopen)[^\n]*oracle", txt):
                    bad.append(os.path.join(dp, f))
    assert not bad, bad


def test_fuse_report_binding_matches_the_library_struct():
    import ctypes as C
    from scannet_b200 import fuse
    from scannet_b200._lib import lib
    lib().scn_fuse_report_sizeof.restype = C.c_size_t
    assert lib().scn_fuse_report_sizeof() == C.sizeof(fuse.FuseReport)


def test_fuse_rejects_a_misspelt_parameter_before_running(built, monkeypatch):
    """a keyword that is no field of scn_tsdf_params raises instead of fusing with the default"""
    import pytest
    from scannet_b200 import fuse

    def driver_must_not_run():
        raise AssertionError("the fusion driver was called")
    monkeypatch.setattr(fuse, "lib", driver_must_not_run)
    with pytest.raises(AttributeError, match="max_block"):
        fuse.fuse_scene("scene.sens", max_block=1 << 20)
    with pytest.raises(AttributeError, match="max_block"):
        fuse.fuse_many(["scene.sens"], max_block=1 << 20)
