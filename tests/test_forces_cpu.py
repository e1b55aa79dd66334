"""External forces and wind without a GPU: the ctypes prototypes of the three entry points against the header, and how
the Python methods shape their arguments (checked against a recording stand-in for the library)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# C parameter type -> the ctypes type the binding must use for it (arrays go through void*, so a null array can be passed)
_C_TO_CTYPES = {"PiesB200Solver*": C.c_void_p, "uint32_t": C.c_uint32, "const uint32_t*": C.c_void_p,
                "const float*": C.c_void_p, "float*": C.c_void_p, "float": C.c_float}


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


def test_force_prototypes_match_header(pb):
    for name, nparams in (("pies_b200_set_external_forces", 4), ("pies_b200_set_wind", 4),
                          ("pies_b200_get_external_forces", 2)):
        ret, params = _prototype(name)
        assert ret == "int" and len(params) == nparams, (name, params)
        res, args = pb.solver._SIGNATURES[name]
        assert res is C.c_int
        assert args == [_C_TO_CTYPES[p] for p in params], (name, params)


class _Recorder:
    """Stands in for the loaded library: records what the methods pass and copies the arrays behind the pointers."""

    def __init__(self, n):
        self.n, self.calls = n, []

    @staticmethod
    def _read(ptr, dtype, count):
        if ptr is None:
            return None
        addr = ptr.value if isinstance(ptr, C.c_void_p) else C.cast(ptr, C.c_void_p).value
        return np.ctypeslib.as_array((np.ctypeslib.as_ctypes_type(dtype) * count).from_address(addr)).copy()

    def pies_b200_set_external_forces(self, h, n, nodes, forces):
        self.calls.append(("forces", n, self._read(nodes, np.uint32, n), self._read(forces, np.float32, 3 * n)))
        return 0

    def pies_b200_set_wind(self, h, velocity, cn, ct):
        self.calls.append(("wind", self._read(velocity, np.float32, 3), cn, ct))
        return 0

    def pies_b200_vertex_count(self, h):
        return self.n

    def pies_b200_get_external_forces(self, h, xyz):
        addr = C.cast(xyz, C.c_void_p).value
        out = np.ctypeslib.as_array((C.c_float * (3 * self.n)).from_address(addr))
        out[:] = np.arange(3 * self.n, dtype=np.float32)
        self.calls.append(("get",))
        return 0


@pytest.fixture
def fake(pb, monkeypatch):
    rec = _Recorder(4)
    monkeypatch.setattr(pb.solver, "_lib", rec)
    s = object.__new__(pb.Solver)   # no device: only the argument shaping runs
    s.h = None
    yield s, rec
    s.h = None


def test_set_external_forces_shaping(pb, fake):
    s, rec = fake
    s.setExternalForces([3, 1], [[1, 2, 3], [4.5, 5, 6]])
    kind, n, ids, f = rec.calls[-1]
    assert kind == "forces" and n == 2
    assert ids.dtype == np.uint32 and ids.tolist() == [3, 1]
    assert f.dtype == np.float32 and f.tolist() == [1, 2, 3, 4.5, 5, 6]
    s.setExternalForces(np.int64([2]), np.float64([7, 8, 9]))   # one node: a flat 3-vector is accepted
    assert rec.calls[-1][1] == 1 and rec.calls[-1][3].tolist() == [7, 8, 9]
    s.setExternalForces([], np.zeros((0, 3)))                    # removal: n = 0 and null arrays
    assert rec.calls[-1] == ("forces", 0, None, None)
    with pytest.raises(ValueError):
        s.setExternalForces([0, 1], [[1, 2, 3]])
    with pytest.raises(ValueError):
        s.setExternalForces([0], [1, 2, 3, 4, 5, 6])


def test_set_wind_and_readback_shaping(pb, fake):
    s, rec = fake
    s.setWind((1, -2, 0.5), 2.0, 0.25)
    kind, v, cn, ct = rec.calls[-1]
    assert kind == "wind" and v.dtype == np.float32 and v.tolist() == [1, -2, 0.5] and (cn, ct) == (2.0, 0.25)
    with pytest.raises(ValueError):
        s.setWind((1, 2), 1.0, 0.0)
    f = s.externalForces()
    assert f.dtype == np.float32 and f.shape == (4, 3)
    assert f.reshape(-1).tolist() == list(range(12))
