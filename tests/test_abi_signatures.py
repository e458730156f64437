"""The ctypes signature table (``_cabi.SIGNATURES``) against the prototypes of ``include/msda_b200.h``.

ctypes does not check argument widths: a ``c_int32`` where the header says ``int64_t``, or a missing ``c_double``,
passes every CPU check and corrupts the arguments only on the GPU. Each table entry must have the prototype's
argument count and, position by position, the same class of type.
"""
import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

_C_SCALARS = {"void": "void", "int": "int32", "int32_t": "int32", "int64_t": "int64", "size_t": "size_t",
              "float": "float", "double": "double"}
_CTYPES_SCALARS = {ctypes.c_int32: "int32", ctypes.c_int64: "int64", ctypes.c_size_t: "size_t",
                   ctypes.c_float: "float", ctypes.c_double: "double"}


def _c_class(decl: str) -> str:
    """Class of one C type (a return type, or a parameter without its name)."""
    if "*" in decl:
        return "pointer"
    words = [w for w in decl.split() if w != "const"]
    assert len(words) == 1 and words[0] in _C_SCALARS, f"unexpected C type {decl!r}"
    return _C_SCALARS[words[0]]


def _ctypes_class(t) -> str:
    if t is None:
        return "void"
    if t in (ctypes.c_void_p, ctypes.c_char_p) or issubclass(t, ctypes._Pointer):
        return "pointer"
    return _CTYPES_SCALARS.get(t, f"unexpected ctypes type {t.__name__}")


@pytest.fixture(scope="module")
def prototypes():
    """name -> (return class, [argument classes]) of every function the header declares."""
    text = open(os.path.join(ROOT, "include", "msda_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"^\s*#.*$", "", text, flags=re.M)
    out = {}
    for ret, name, args in re.findall(r"([^;{}]*?)\b(msda_b200_\w+)\s*\(([^)]*)\)\s*;", text):
        params = [] if args.strip() in ("", "void") else [p.strip() for p in args.split(",")]
        arg_classes = []
        for p in params:
            pointer = "*" in p
            decl = p[:p.rfind("*") + 1] if pointer else p.rsplit(None, 1)[0]  # drop the parameter's name
            arg_classes.append(_c_class(decl))
        out[name] = (_c_class(" ".join(ret.split())), arg_classes)
    return out


def test_table_covers_the_header(prototypes):
    from weed_instance_segmentation_b200 import _cabi
    assert len(prototypes) == 37
    assert sorted(_cabi.SIGNATURES) == sorted(prototypes)
    assert _cabi.EXPORTS == tuple(_cabi.SIGNATURES)
    assert prototypes["msda_b200_last_error"] == ("pointer", [])  # const char* return
    assert "double" in prototypes["msda_b200_postprocess_paint"][1]


def test_table_matches_header_prototypes(prototypes):
    from weed_instance_segmentation_b200 import _cabi
    bad = []
    for name, (restype, argtypes) in _cabi.SIGNATURES.items():
        want_ret, want_args = prototypes[name]
        got_args = [_ctypes_class(t) for t in argtypes]
        if _ctypes_class(restype) != want_ret:
            bad.append(f"{name}: returns {_ctypes_class(restype)}, header {want_ret}")
        if got_args != want_args:
            bad.append(f"{name}: arguments {got_args}, header {want_args}")
    assert not bad, "\n".join(bad)
