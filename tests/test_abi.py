"""The C-ABI library builds for sm_100a, loads, and exports every symbol the header declares
(no compute calls: this runs without a GPU)."""
import ctypes
import os
import re

from mobrob_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "mobrob_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mr_[a-z0-9_]+)\s*\(", text)))


_C_KINDS = {"int": "int", "int32_t": "int", "unsigned": "unsigned", "int64_t": "int64_t", "uint64_t": "uint64_t",
            "float": "float", "double": "double", "void": None}
_CTYPES_KINDS = {ctypes.c_int: "int", ctypes.c_uint: "unsigned", ctypes.c_int64: "int64_t",
                 ctypes.c_uint64: "uint64_t", ctypes.c_float: "float", ctypes.c_double: "double", None: None}


def _c_kind(decl):
    """Kind of a parameter or return declaration: "pointer" or the scalar type with const and the name dropped."""
    if "*" in decl:
        return "pointer"
    words = [w for w in decl.split() if w != "const"]
    return _C_KINDS[words[0]]


def _ctypes_kind(t):
    if t in (ctypes.c_void_p, ctypes.c_char_p) or (isinstance(t, type) and issubclass(t, ctypes._Pointer)):
        return "pointer"
    return _CTYPES_KINDS[t]


def _header_prototypes():
    """{name: (return kind, [parameter kinds])} of every prototype in the comment-stripped header."""
    text = open(os.path.join(ROOT, "include", "mobrob_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = "\n".join(line for line in text.splitlines() if not line.lstrip().startswith("#"))
    protos = {}
    for ret, name, params in re.findall(r"(?:^|(?<=[;{}]))\s*([^;{}()]*?)\b(mr_\w+)\s*\(([^()]*)\)\s*;", text):
        params = [p for p in (p.strip() for p in params.split(",")) if p and p != "void"]
        protos[name] = (_c_kind(ret), [_c_kind(p) for p in params])
    return protos


def test_ctypes_signatures_match_header_prototypes():
    """Every _SIGNATURES row has the arity and the argument kinds of its C prototype: a row out of step with the
    header would pass garbage to a kernel as a pointer, so it must fail here, without a GPU."""
    protos = _header_prototypes()
    assert sorted(protos) == _header_symbols()
    for name, (ret, params) in protos.items():
        res, args = _lib._SIGNATURES[name]
        got = [_ctypes_kind(a) for a in args]
        assert len(got) == len(params), f"{name}: header has {len(params)} parameters, _SIGNATURES {len(got)}"
        assert got == params, f"{name}: header {params} != _SIGNATURES {got}"
        assert _ctypes_kind(res) == ret, f"{name}: header returns {ret}, _SIGNATURES {_ctypes_kind(res)}"


def test_library_builds_and_exports_header():
    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    syms = _header_symbols()
    assert len(syms) >= 15
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/mobrob_b200.h but not exported"
    assert sorted(_lib.exported_symbols()) == syms, "ctypes table and header are out of sync"


def test_version_and_error_string():
    lib = _lib.load()
    assert lib.mr_version() >= 100
    assert isinstance(lib.mr_last_error(), bytes)
    assert lib.mr_launch_count() >= 0


def test_bad_arguments_fail_loudly_without_gpu():
    lib = _lib.load()
    h = ctypes.c_void_p()
    assert lib.mr_env_create(7, 4, 0, 1000, 1, ctypes.byref(h)) != 0
    assert b"kind" in lib.mr_last_error()
    assert lib.mr_env_create(0, 0, 0, 1000, 1, ctypes.byref(h)) != 0
