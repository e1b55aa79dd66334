"""The fused local step + RHS (`k_tet_rhs`, one CTA per closed segment) against the two-kernel path it replaces
(`k_tet_elems` then `k_gather_rhs[_contacts]`, forced with PIES_B200_NO_FUSED_LOCAL): the same projection code and
the same order of float adds, so the trajectories must agree bit for bit, through the first impacts and the stacking.
The switch is read once per process, so each path runs in its own subprocess."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCENES = {
    # four columns of twelve S3 bodies: free fall, first impacts from tick ≈ 20, stacked columns after
    "s3_stack": "scenes.build_s3(s, bodies=48, nx=2, nz=2)",
    # segments cut by a distance-constraint sheet and a shape-matching box (both on the two-kernel path)
    "mixed": ("[s.createTetBox((3.0 * i, 0.6, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(3)]\n"
              "s.createSheet((0.0, 4.0, 0.0), 1.0, 1.0, 1000.0)\n"
              "[s.createTetBox((3.0 * i, 2.6, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(7)]\n"
              "s.createShapeMatchingBox((10.0, 1.0, 0.0), 3, 4, 4, 0.5, (0, 0, 0), 1000.0)\n"
              "[s.createTetBox((3.0 * i, 5.0, 3.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(2)]"),
    # a TetGen cube over the segment cap (two-kernel path) dropping on the floor next to tet boxes (fused)
    "tetgen_cube": ("pts, tets, faces = scenes.cube24_mesh()\n"
                    "s.addTetMeshVolume(pts + np.float32([0.0, 0.3, 0.0]), tets, faces, (0, 0, 0), 1.0, 1000.0, 0.8, 1.0, 1000.0, 1.0, 1.0)\n"
                    "[s.createTetBox((10.0 + 3.0 * i, 1.0, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(4)]"),
}
TICKS = 48
CHECK = (1, 10, 20, 30, 40, 48)

SCRIPT = """import sys; sys.path.insert(0, %r)
import numpy as np
import pies_b200 as pb
from pies_b200 import scenes
s = pb.Solver(**scenes.S3_OPTIONS)
%s
out, launches, contacts = {}, [], []
for t in range(1, %d + 1):
    s.tick()
    st = s.stats()
    launches.append(st.kernelLaunchesLastTick); contacts.append((st.triCollisions, st.staticCollisions))
    if t in %r:
        out["pos%%d" %% t], out["prev%%d" %% t], out["vel%%d" %% t] = s.positions, s.prevPositions, s.velocities
np.savez(sys.argv[1], launches=np.array(launches), contacts=np.array(contacts), failed=np.array(s.simFailed), **out)
"""


def _run(scene, path, fused):
    env = dict(os.environ)
    env.pop("PIES_B200_NO_FUSED_LOCAL", None)
    if not fused:
        env["PIES_B200_NO_FUSED_LOCAL"] = "1"
    subprocess.run([sys.executable, "-c", SCRIPT % (ROOT, SCENES[scene], TICKS, CHECK), str(path)], check=True, env=env)
    return np.load(path)


@pytest.mark.parametrize("scene", sorted(SCENES))
def test_fused_local_step_is_bit_identical(pb, scene, tmp_path):
    a = _run(scene, tmp_path / "fused.npz", True)
    b = _run(scene, tmp_path / "two_kernel.npz", False)
    assert not a["failed"] and not b["failed"]
    assert a["contacts"][:, 0].max() > 0 or a["contacts"][:, 1].max() > 0   # the window reaches contact
    for t in CHECK:
        for k in ("pos", "prev", "vel"):
            assert np.isfinite(a["%s%d" % (k, t)]).all()
            assert np.array_equal(a["%s%d" % (k, t)], b["%s%d" % (k, t)]), (scene, k, t)
    assert np.array_equal(a["contacts"], b["contacts"])
    # the fused path really ran (10 PD iterations per tick): k_tet_rhs replaces k_tet_elems + gather where every body is
    # in a segment, replaces k_tet_elems where no tet is residual, and runs next to both where tets are residual too
    delta = a["launches"].astype(np.int64) - b["launches"].astype(np.int64)
    assert (delta == {"s3_stack": -10, "mixed": 0, "tetgen_cube": 10}[scene]).all(), (scene, np.unique(delta))
