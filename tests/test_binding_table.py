"""The ctypes binding table (_lib.BINDINGS) against every DCN_API prototype of include/dcn_b200.h.

A binding with one argument too few or of the wrong kind shifts every argument after it, which the library only
notices as a device fault; this compares the table with the header as plain data, without a built library."""
import ctypes
import os
import re

import pytest

from jittor_dcn_b200 import _lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = ("DcnShape", "DcnMsdaShape", "DcnV3Shape")


def _prototypes():
    """{export name: (return C type, [parameter C types])} of every DCN_API declaration in the header."""
    text = open(os.path.join(ROOT, "include", "dcn_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", " ", text, flags=re.S)
    protos = {}
    for ret, name, params in re.findall(r"DCN_API\s+([^;(]*?)\s*\b(dcn_\w+)\s*\(([^)]*)\)\s*;", text):
        params = [p.strip() for p in params.split(",")]
        if params == ["void"]:
            params = []
        # drop each parameter's name: what is left is its type
        protos[name] = (ret, [re.match(r"(.*?)\w+$", p, re.S).group(1) for p in params])
    return protos


PROTOTYPES = _prototypes()


def _c_kind(ctype):
    t = re.sub(r"\bconst\b|\s", "", ctype)
    if t.endswith("*") and t[:-1] in SHAPES:
        return t[:-1]
    if t.endswith("*"):
        return "pointer"
    # size_t and uint64_t are one ctypes type (c_ulong) on LP64
    return {"int": "int", "int32_t": "int", "float": "float", "size_t": "u64", "uint64_t": "u64", "void": "void"}[t]


def _ctypes_kind(t):
    if t is None:
        return "void"
    if issubclass(t, ctypes._Pointer) and issubclass(t._type_, ctypes.Structure):
        return t._type_.__name__
    if t in (ctypes.c_void_p, ctypes.c_char_p) or issubclass(t, ctypes._Pointer):
        return "pointer"
    return {ctypes.c_int32: "int", ctypes.c_float: "float", ctypes.c_uint64: "u64"}.get(t, t.__name__)


def test_every_declared_export_is_bound_and_every_binding_is_declared():
    assert sorted(set(PROTOTYPES) - set(_lib.BINDINGS)) == [], "declared in include/dcn_b200.h but not bound"
    assert sorted(set(_lib.BINDINGS) - set(PROTOTYPES)) == [], "bound but not declared in include/dcn_b200.h"
    assert _lib.EXPORTS == tuple(_lib.BINDINGS)


@pytest.mark.parametrize("name", sorted(PROTOTYPES))
def test_binding_matches_the_prototype(name):
    ret, params = PROTOTYPES[name]
    restype, argtypes = _lib.BINDINGS[name]
    assert _ctypes_kind(restype) == _c_kind(ret), f"{name} returns {ret}"
    assert len(argtypes) == len(params), f"{name} takes {len(params)} parameters: {params}"
    for i, (t, p) in enumerate(zip(argtypes, params)):
        assert _ctypes_kind(t) == _c_kind(p), f"{name} parameter {i} is {p}"
