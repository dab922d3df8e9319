"""CPU: the C-ABI library builds for sm_100a, loads, and exports every symbol include/crfconv_b200.h declares.
No compute calls (there is no GPU here)."""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def built():
    from crfconv_b200 import build
    return build.build()


def _header():
    src = open(os.path.join(ROOT, "include", "crfconv_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return re.sub(r"//[^\n]*", "", src)


def _declared():
    return sorted(set(re.findall(r"\b(crfconv_[a-z0-9_]+)\s*\(", _header())))


_SCALARS = ("int", "int64_t", "size_t", "uint32_t", "float")


def _kind(decl):
    """Kind of a C parameter or return type: 'pointer' or one of _SCALARS ('const float* X' -> 'pointer', 'int64_t M' -> 'int64_t')."""
    if "*" in decl:
        return "pointer"
    typ = decl.split()[0]
    assert typ in _SCALARS, f"unexpected C type in {decl!r}"
    return typ


def _prototypes():
    """name -> (return kind, [argument kinds]) for every prototype of the header."""
    out = {}
    for ret, name, args in re.findall(r"((?:const\s+)?\w+\s*\**)\s*\b(crfconv_[a-z0-9_]+)\s*\(([^)]*)\)\s*;", _header()):
        args = " ".join(args.split())
        out[name] = (_kind(ret), [] if args in ("", "void") else [_kind(a.strip()) for a in args.split(",")])
    return out


def test_library_exports_every_declared_symbol(built):
    h = ctypes.CDLL(built)
    names = _declared()
    assert len(names) >= 8
    for n in names:
        assert hasattr(h, n), f"{n} declared in include/crfconv_b200.h but not exported"


def test_python_signature_table_matches_header(built):
    """Names, argument counts and argument kinds: ctypes forwards surplus arguments silently, so one stray `int` in _lib would
    shift every later argument of a call without any error on the host."""
    from crfconv_b200 import _lib
    assert sorted(_lib.SIGNATURES) == _declared()
    protos = _prototypes()
    assert sorted(protos) == _declared()
    kind = {ctypes.c_void_p: "pointer", ctypes.c_char_p: "pointer", ctypes.c_int: "int", ctypes.c_int64: "int64_t",
            ctypes.c_size_t: "size_t", ctypes.c_uint32: "uint32_t", ctypes.c_float: "float"}
    for name, (res, args) in _lib.SIGNATURES.items():
        assert (kind[res], [kind[a] for a in args]) == protos[name], name
    assert _lib.lib().crfconv_abi_version() == 2
    assert _lib.lib().crfconv_status_string(-2) == b"workspace too small"


def test_workspace_queries_run_without_a_gpu(built):
    from crfconv_b200 import _lib
    L = _lib.lib()
    assert L.crfconv_knn_workspace_bytes(2, 40960, 40960, 16) > 2 * 40960 * 16
    assert L.crfconv_grid_subsample_workspace_bytes(100000, 3, 1) > 100000 * 24


def test_product_never_imports_the_oracle():
    """The product package must not reference oracle/ (tier rule ③)."""
    pkg = os.path.join(ROOT, "crfconv_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, flags=re.M), f
                assert "oracle/" not in txt and "liboracle" not in txt, f


def test_no_silent_fallback_when_library_missing(monkeypatch, tmp_path):
    from crfconv_b200 import _lib
    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU"):
        _lib.lib()
