"""CPU test of build.py: the library is rebuilt whenever a file it is compiled from changes."""
import importlib.util
import os
import shutil

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "extendedrtirtmodeling.jl_b200")


def _build_module():
    spec = importlib.util.spec_from_file_location("erirt_b200_build_under_test", os.path.join(PKG, "build.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_every_csrc_file_is_a_dependency_of_the_library(tmp_path, monkeypatch):
    """A copy of csrc/ and include/ with a library newer than all of it: touching any one file makes is_stale() true."""
    B = _build_module()
    pkg = tmp_path / "pkg"
    shutil.copytree(os.path.join(PKG, "csrc"), pkg / "csrc")
    shutil.copytree(os.path.join(ROOT, "include"), tmp_path / "include")
    lib = pkg / "liberirt_b200.so"
    lib.write_bytes(b"")
    monkeypatch.setattr(B, "HERE", str(pkg))
    monkeypatch.setattr(B, "CSRC", str(pkg / "csrc"))
    monkeypatch.setattr(B, "LIB", str(lib))
    files = sorted(os.listdir(pkg / "csrc"))
    assert "erirt_b200.cu" in files and "diagnostics.cuh" in files
    deps = [pkg / "csrc" / f for f in files] + [tmp_path / "include" / "erirt_b200.h"]
    old, built, new = 1_000_000, 2_000_000, 3_000_000
    for d in deps:
        os.utime(d, (old, old))
    os.utime(lib, (built, built))
    assert not B.is_stale()
    for d in deps:
        os.utime(d, (new, new))
        assert B.is_stale(), f"{d.name} changed but the library is not rebuilt"
        os.utime(d, (old, old))
