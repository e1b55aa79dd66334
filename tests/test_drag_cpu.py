"""Drag targets and the raycast without a GPU: the ctypes prototypes of the two entry points against the header."""
import ctypes as C
import os
import re

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# C parameter type -> the ctypes type the binding must use for it (arrays go through void*, so a null array can be passed)
_C_TO_CTYPES = {"PiesB200Solver*": C.c_void_p, "uint32_t": C.c_uint32, "const uint32_t*": C.c_void_p,
                "const float*": C.c_void_p, "int32_t*": C.c_void_p, "float*": C.c_void_p}


def _prototype(name):
    text = open(os.path.join(ROOT, "include", "pies_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    m = re.search(r"(\w+)\s+%s\s*\((.*?)\);" % name, text, re.S)
    assert m, name
    params = []
    for p in m.group(2).split(","):
        p = " ".join(p.split())
        params.append(re.sub(r"\s*\w+$", "", p).replace(" *", "*"))
    return m.group(1), params


def test_drag_and_raycast_prototypes_match_header(pb):
    for name, nparams in (("pies_b200_set_drag_targets", 5), ("pies_b200_raycast", 8)):
        ret, params = _prototype(name)
        assert ret == "int" and len(params) == nparams, (name, params)
        res, args = pb.solver._SIGNATURES[name]
        assert res is C.c_int
        assert args == [_C_TO_CTYPES[p] for p in params], (name, params)
