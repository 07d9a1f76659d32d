"""The C-ABI library builds for sm_100a, loads, and exports every symbol include/dks.h declares.  No compute here."""
import ctypes
import os
import re

import pytest

from distributedkernelshap_b200 import _cabi, build

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(REPO, "include", "dks.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(dks_[a-z0-9_]+)\s*\(", text)))


def test_library_builds_and_exports_declared_symbols():
    if build.find_nvcc() is None and not os.path.exists(build.LIB_PATH):
        pytest.skip("no nvcc and no prebuilt library")
    lib = _cabi.load()
    names = declared_symbols()
    assert len(names) >= 25
    for name in names:
        assert hasattr(lib, name), f"{name} declared in dks.h but not exported"
        assert name in _cabi.SIGNATURES, f"{name} has no ctypes signature"
    assert set(_cabi.SIGNATURES) == set(names)
    assert lib.dks_version() == 100


def test_sass_is_sm100a():
    nvcc = build.find_nvcc()
    if nvcc is None:
        pytest.skip("no CUDA toolkit")
    import subprocess
    _cabi.load()
    cuobjdump = os.path.join(os.path.dirname(nvcc), "cuobjdump")     # the toolkit's bin directory need not be on PATH
    out = subprocess.run([cuobjdump, "-lelf", build.LIB_PATH], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_no_cpu_fallback_without_a_gpu():
    lib = _cabi.load()
    n = ctypes.c_int(-1)
    assert lib.dks_device_count(ctypes.byref(n)) == 0
    if n.value > 0:
        pytest.skip("a GPU is present")
    ctx = ctypes.c_void_p()
    rc = lib.dks_create(ctypes.byref(ctx), 0)
    assert rc == _cabi.DKS_ERR_CUDA and b"no CPU fallback" in lib.dks_last_error()
    from distributedkernelshap_b200.engine import GpuKernelExplainer
    from conftest import make_problem
    prob = make_problem()
    with pytest.raises(_cabi.DksError):
        GpuKernelExplainer(prob["clf"].predict_proba, prob["bg"], link="logit")


def test_product_does_not_import_the_oracle():
    pkg = os.path.join(REPO, "distributedkernelshap_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"
                assert "shap_kernel_oracle" not in src, f"{f} references the oracle module"
