"""The C-ABI library loads without a GPU and exports exactly what include/unite_b200.h declares."""
import os
import re
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_functions():
    src = open(os.path.join(ROOT, "include", "unite_b200.h")).read()
    return sorted(set(re.findall(r"UB_API\s+[\w\s\*]+?\b(ub_\w+)\s*\(", src)))


def test_library_loads_and_reports_version():
    from unite_b200 import _cabi
    assert _cabi.lib.ub_version() >= 100
    assert _cabi.lib.ub_last_error() is not None


def test_every_declared_symbol_is_exported_and_bound():
    from unite_b200 import _cabi
    declared = _header_functions()
    assert len(declared) >= 20
    out = subprocess.run(["nm", "-D", "--defined-only", _cabi._LIB_PATH], capture_output=True, text=True, check=True).stdout
    exported = sorted(set(re.findall(r" T (ub_\w+)", out)))
    assert exported == declared, (set(declared) ^ set(exported))
    assert sorted(_cabi.SIGNATURES) == declared


def test_erf_build_exports_the_same_abi():
    """build() also produces libunite_b200_erf.so (-DUB_GELU_ERF): the same exported symbols as the default library."""
    from unite_b200 import _cabi
    declared = _header_functions()
    path = os.path.join(os.path.dirname(_cabi._LIB_PATH), "libunite_b200_erf.so")
    assert os.path.exists(path), f"build() did not produce {path}"
    out = subprocess.run(["nm", "-D", "--defined-only", path], capture_output=True, text=True, check=True).stdout
    assert sorted(set(re.findall(r" T (ub_\w+)", out))) == declared


def test_sass_uses_blackwell_tensor_and_tma_paths():
    from unite_b200 import _cabi
    r = subprocess.run(["cuobjdump", "-sass", _cabi._LIB_PATH], capture_output=True, text=True)
    if r.returncode != 0:
        import pytest
        pytest.skip("cuobjdump not available")
    assert "UTCHMMA" in r.stdout and "UTMALDG" in r.stdout and "LDTM" in r.stdout
    # every tensor-core product is a tcgen05 MMA (UTCHMMA): no kernel uses the older warp-level mma.sync (plain HMMA)
    assert not re.search(r"(?<!UTC)HMMA\.", r.stdout)


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "unite_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, re.M), f
