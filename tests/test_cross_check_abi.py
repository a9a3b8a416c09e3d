"""Without a GPU: the cross-check entry points are exported and their ctypes prototypes match include/cvgraft.h."""
import ctypes as C
import os
import re

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))

# C parameter type in the header -> ctypes type the prototype must use
_CTYPE = {"cvg_ctx*": C.c_void_p, "const cvg_models*": C.c_void_p, "int": C.c_int, "const float*": C.c_void_p,
          "int32_t*": C.c_void_p, "float*": C.c_void_p}


def _header_params(name):
    hdr = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "cvgraft.h")).read(), flags=re.S)
    m = re.search(r"\bint\s+" + name + r"\s*\(([^)]*)\)\s*;", hdr)
    assert m, name
    return [re.sub(r"\s*\b\w+$", "", p.strip()).replace(" *", "*") for p in m.group(1).split(",")]


def test_cross_check_symbols_and_prototypes():
    from computervision_objectdetection_featurematching_b200 import _lib, build
    build.build()
    lib = _lib.load()
    for name in ("cvg_match_cross_check", "cvg_match_cross_check_raw"):
        assert hasattr(lib, name)
        res, args = _lib.SYMBOLS[name]
        assert res is C.c_int
        assert args == [_CTYPE[p] for p in _header_params(name)], name
