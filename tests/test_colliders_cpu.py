"""Static colliders without a GPU: the ctypes mirror of PiesB200Collider against the header, and the Python helpers."""
import ctypes as C
import os
import re

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_collider_layout_matches_header(pb):
    assert C.sizeof(pb.Collider) == 64
    offsets = {name: getattr(pb.Collider, name).offset for name, _ in pb.Collider._fields_}
    assert offsets == {"kind": 0, "center": 4, "axes": 16, "extent": 52}
    text = open(os.path.join(ROOT, "include", "pies_b200.h")).read()
    body = re.search(r"typedef struct PiesB200Collider \{(.*?)\} PiesB200Collider;", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    fields = re.findall(r"(uint32_t|float)\s+(\w+)(?:\[(\d+)\])?;", body)
    assert [(f[1], int(f[2] or 1)) for f in fields] == [("kind", 1), ("center", 3), ("axes", 9), ("extent", 3)]
    kinds = dict(re.findall(r"#define PIES_B200_COLLIDER_(\w+) (\d+)", text))
    assert {k: int(v) for k, v in kinds.items()} == {"HALFSPACE": pb.solver.COLLIDER_HALFSPACE,
                                                      "SPHERE": pb.solver.COLLIDER_SPHERE, "BOX": pb.solver.COLLIDER_BOX}
    assert int(re.search(r"#define PIES_B200_MAX_COLLIDERS (\d+)", text).group(1)) == pb.solver.MAX_COLLIDERS == 32


def test_halfspace_helper_normalises(pb):
    c = pb.halfspace((1.0, 2.0, 3.0), (0.0, 3.0, 4.0))
    assert c.kind == pb.solver.COLLIDER_HALFSPACE
    assert list(c.center) == [1.0, 2.0, 3.0]
    assert np.allclose(list(c.axes)[:3], [0.0, 0.6, 0.8], atol=1e-7)
    assert list(c.axes)[3:] == [0.0] * 6
    z = pb.halfspace((0, 0, 0), (0, 0, 0))   # left for the library to reject
    assert list(z.axes)[:3] == [0.0, 0.0, 0.0]


def test_sphere_and_box_helpers(pb):
    s = pb.sphere((0.5, 1.0, -2.0), 0.75)
    assert s.kind == pb.solver.COLLIDER_SPHERE and list(s.center) == [0.5, 1.0, -2.0] and s.extent[0] == 0.75
    b = pb.box((1, 2, 3), (0.5, 1.0, 1.5))
    assert b.kind == pb.solver.COLLIDER_BOX
    assert list(b.axes) == [1, 0, 0, 0, 1, 0, 0, 0, 1] and list(b.extent) == [0.5, 1.0, 1.5]
    c, s_ = np.cos(0.3), np.sin(0.3)
    R = np.array([[c, -s_, 0.0], [s_, c, 0.0], [0.0, 0.0, 1.0]])   # columns = the box's axes
    r = pb.box((0, 0, 0), (1, 1, 1), R)
    assert np.allclose(np.array(list(r.axes)).reshape(3, 3), R.T, atol=1e-7)   # stored column after column
