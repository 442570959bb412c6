"""The C-ABI library loads on a CPU-only box and exports every symbol include/qsb200.h declares.
No compute entry point is called here (there is no GPU and no CPU fallback)."""

import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "qsb200.h")


def declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(qs_[a-z0-9_]+)\s*\(", text)))


@pytest.fixture(scope="module")
def library():
    from quantum_systems_b200 import _native
    from quantum_systems_b200.build import build

    build()
    return _native.load()


def test_header_and_binding_agree(library):
    from quantum_systems_b200 import _native

    names = declared_functions()
    assert len(names) >= 20
    assert sorted(_native.SIGNATURES) == names
    # a stale argtypes list is not caught at compile time: ctypes would pass the arguments shifted
    text = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    prototypes = dict(re.findall(r"\b(qs_[a-z0-9_]+)\s*\(([^()]*)\)\s*;", text))
    assert sorted(prototypes) == names
    for name, params in prototypes.items():
        count = 0 if params.strip() in ("", "void") else params.count(",") + 1
        assert count == len(_native.SIGNATURES[name]), f"{name}: {count} parameters in the header"


def test_every_declared_symbol_is_exported(library):
    raw = ctypes.CDLL(os.path.join(ROOT, "quantum_systems_b200", "libqsb200.so"))
    for name in declared_functions():
        assert hasattr(raw, name), f"{name} declared in include/qsb200.h but not exported"


def test_version_and_argument_validation(library):
    assert library.qs_version() >= 100
    nbytes = ctypes.c_int64(-1)
    # host-only planning calls work without a device
    assert library.qs_transform_two_body_workspace_bytes(128, 128, 0, 0, ctypes.byref(nbytes)) == 0
    assert nbytes.value >= 2 * 8 * 128**4
    assert library.qs_coeff_image_bytes(0, 4, 0, 0, ctypes.byref(nbytes)) != 0
    assert b"bad arguments" in library.qs_last_error()


def test_product_package_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "quantum_systems_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(".py"):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the oracle", ""), f"{f} mentions the oracle package"


def test_cpu_tensor_has_no_fallback():
    torch = pytest.importorskip("torch")
    from quantum_systems_b200 import ops

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        ops.transform_two_body(torch.zeros((2,) * 4, dtype=torch.float64), torch.eye(2, dtype=torch.float64))
