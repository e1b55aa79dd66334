"""Static colliders (half-spaces, spheres, oriented boxes) in the PD and PBD ticks, DESIGN.md section 9."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
W = 1.0e4   # the weight of a node-collider contact (the floor's StaticCollisionConstraint::w)


# ---- float64 restatement of phi and n (include/pies_b200.h) ------------------------------------------------------
def np_phi(c, x):
    """(phi[N], n[N, 3]) of one Collider at points x[N, 3], in float64, with the documented tie rules."""
    x = np.asarray(x, np.float64).reshape(-1, 3)
    ctr = np.array(list(c.center), np.float64)
    ax = np.array(list(c.axes), np.float64)
    ext = np.array(list(c.extent), np.float64)
    d = x - ctr
    if c.kind == 0:
        n = ax[:3] / np.linalg.norm(ax[:3])
        return d @ n, np.broadcast_to(n, x.shape).copy()
    if c.kind == 1:
        ln = np.linalg.norm(d, axis=1)
        n = np.where(ln[:, None] > 0, d / np.where(ln > 0, ln, 1.0)[:, None], np.array([0.0, 1.0, 0.0]))
        return ln - ext[0], n
    A = ax.reshape(3, 3)               # row a = axis a
    loc = d @ A.T
    q = np.abs(loc) - ext
    out = (q > 0).any(axis=1)
    o = np.where(q > 0, np.sign(loc) * q, 0.0)
    ln = np.linalg.norm(o, axis=1)
    phi = np.where(out, ln, q.max(axis=1))
    nl = np.zeros_like(x)
    nl[out] = o[out] / ln[out, None]
    a = np.argmax(q, axis=1)           # first maximum = the lowest axis on a tie
    sgn = np.where(loc[np.arange(len(x)), a] < 0, -1.0, 1.0)
    ins = ~out
    nl[ins, a[ins]] = sgn[ins]
    return phi, nl @ A


def np_project(c, x):
    phi, n = np_phi(c, x)
    return x - np.minimum(phi, 0.0)[:, None] * n


def bin_walls(pos, margin, pb, floor=False):
    lo, hi = pos.min(0) - margin, pos.max(0) + margin
    walls = [pb.halfspace((lo[0], 0, 0), (1, 0, 0)), pb.halfspace((hi[0], 0, 0), (-1, 0, 0)),
             pb.halfspace((0, 0, lo[2]), (0, 0, 1)), pb.halfspace((0, 0, hi[2]), (0, 0, -1))]
    if floor:
        walls.append(pb.halfspace((0, 0, 0), (0, 1, 0)))
    return walls


# ---- 1. no behaviour change --------------------------------------------------------------------------------------
SCENES = {
    "s3_stack": "scenes.build_s3(s, bodies=48, nx=2, nz=2)",
    "mixed": ("[s.createTetBox((3.0 * i, 0.6, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(3)]\n"
              "s.createSheet((0.0, 4.0, 0.0), 1.0, 1.0, 1000.0)\n"
              "[s.createTetBox((3.0 * i, 2.6, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(7)]\n"
              "s.createShapeMatchingBox((10.0, 1.0, 0.0), 3, 4, 4, 0.5, (0, 0, 0), 1000.0)\n"
              "[s.createTetBox((3.0 * i, 5.0, 3.0), 1.0, (0, 0, 0), 1000.0, 1.0, False) for i in range(2)]"),
}


def _states(pb, build, ticks, pd=True):
    from pies_b200 import scenes  # noqa: F401 (used by the scene strings)
    out = []
    for mode in ("never", "empty", "removed", "untouched"):
        s = pb.Solver(**scenes.S3_OPTIONS) if pd else pb.Solver(solver="PBD")
        build(s)
        if mode == "empty":
            s.setColliders([])
        elif mode == "removed":
            s.setColliders([pb.sphere((0, 0, 0), 5.0)])
            s.setColliders([])
        elif mode == "untouched":
            s.setColliders([pb.sphere((0.0, -500.0, 0.0), 1.0)])
        for _ in range(ticks):
            s.tick()
        assert not s.simFailed
        out.append((mode, s.positions, s.prevPositions, s.velocities))
        s.close()
    return out


@pytest.mark.parametrize("scene", sorted(SCENES))
def test_no_collider_is_bit_identical(pb, scene):
    from pies_b200 import scenes

    def build(s):
        exec(SCENES[scene], {"s": s, "scenes": scenes, "np": np})
    runs = _states(pb, build, 48)
    for mode, *arrs in runs[1:]:
        for a, b in zip(runs[0][1:], arrs):
            assert np.isfinite(a).all()
            assert np.array_equal(a, b), (scene, mode)


def test_no_collider_is_bit_identical_pbd(pb):
    from pies_b200 import scenes
    runs = _states(pb, scenes.build_pbd_boxes, 48, pd=False)
    for mode, *arrs in runs[1:]:
        for a, b in zip(runs[0][1:], arrs):
            assert np.array_equal(a, b), mode


# ---- 2. geometry ---------------------------------------------------------------------------------------------------
def test_probe_matches_float64_restatement(pb):
    rng = np.random.default_rng(7)
    c, s_ = np.cos(0.4), np.sin(0.4)
    R = np.array([[c, 0.0, s_], [0.0, 1.0, 0.0], [-s_, 0.0, c]]) @ np.array([[1.0, 0.0, 0.0], [0.0, np.cos(0.7), -np.sin(0.7)],
                                                                              [0.0, np.sin(0.7), np.cos(0.7)]])
    cols = [pb.halfspace((0.25, -0.5, 1.0), (0.3, 1.0, -0.2)), pb.sphere((0.5, 0.25, -1.0), 1.25),
            pb.box((0.5, 0.25, -1.0), (1.0, 1.0, 1.0)),            # axis-aligned cube: exact ties
            pb.box((-0.3, 0.7, 0.2), (0.5, 1.0, 1.5), R)]
    pts = [rng.uniform(-3, 3, (4000, 3))]
    e = np.array([0.5, 1.0, 1.5])
    for sx in (-1, 0, 1):   # faces, edges, corners of the rotated box, just inside and just outside
        for sy in (-1, 0, 1):
            for sz in (-1, 0, 1):
                for f in (0.9, 1.0, 1.1):
                    pts.append((np.array([-0.3, 0.7, 0.2]) + R @ (f * e * np.array([sx, sy, sz])))[None])
    ctr = np.array([0.5, 0.25, -1.0])
    special = np.array([[0, 0, 0], [0, 0.5, 0], [0, -0.5, 0.5], [1, 0, 0], [1, 1, 0], [2, 2, 2], [2, 2, 0], [-0.5, 0, 0],
                        [0, 0, -0.25]], np.float64) + ctr
    pts.append(special)
    x = np.concatenate(pts).astype(np.float32)
    phi, nrm = pb.probe_colliders(x, cols)
    for k, col in enumerate(cols):
        ref_phi, ref_n = np_phi(col, x.astype(np.float64))
        assert np.allclose(phi[:, k], ref_phi, atol=4e-6, rtol=0), k
        if col.kind == 2:   # normals away from the places where the nearest face switches or the surface is met
            A = np.array(list(col.axes), np.float64).reshape(3, 3)
            q = np.sort(np.abs((x - np.array(list(col.center))) @ A.T) - np.array(list(col.extent)), axis=1)
            ok = (ref_phi > 1e-3) | ((ref_phi < -1e-4) & (q[:, 2] - q[:, 1] > 1e-4))
        else:
            ok = np.linalg.norm(x - np.array(list(col.center)), axis=1) > 1e-3
        assert np.allclose(nrm[ok, k], ref_n[ok], atol=1e-5), k
    # the tie rules and the sphere centre, exactly
    ns = len(special)
    # centre: a three-way tie -> axis 0, + side; (0, -.5, .5): tie of axes 1 and 2 -> axis 1; on a face and on an edge
    assert np.allclose(nrm[-ns:, 2], [[1, 0, 0], [0, 1, 0], [0, -1, 0], [1, 0, 0], [1, 0, 0], [1 / np.sqrt(3)] * 3,
                                      [1 / np.sqrt(2), 1 / np.sqrt(2), 0], [-1, 0, 0], [0, 0, -1]], atol=1e-7)
    assert np.allclose(phi[-ns:, 2], [-1, -0.5, -0.5, 0, 0, np.sqrt(3), np.sqrt(2), -0.5, -0.75], atol=1e-6)
    assert np.array_equal(nrm[-ns, 1], np.float32([0, 1, 0]))   # sphere centre: +y
    assert phi[-ns, 1] == np.float32(-1.25)


# ---- 3. detection --------------------------------------------------------------------------------------------------
def test_detection_masks_match_numpy(pb):
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=48, nx=2, nz=2)
    pos = s.positions
    mid = 0.5 * (pos.min(0) + pos.max(0))
    cols = [pb.halfspace((mid[0], 0, 0), (1, 0, 0)), pb.sphere(mid, 2.0),
            pb.box(mid + np.float32([0, 3.0, 0]), (1.0, 0.7, 2.0), np.array([[0.8, -0.6, 0], [0.6, 0.8, 0], [0, 0, 1]]))]
    s.setColliders(cols)
    s.detect()
    masks = s.colliderContacts()
    thick = s.getOptions().collisionThickness
    expect = np.zeros(len(pos), np.uint32)
    far = np.ones(len(pos), bool)
    for k, c in enumerate(cols):
        phi, _ = np_phi(c, pos)
        expect |= np.where(phi < thick, np.uint32(1 << k), np.uint32(0))
        far &= np.abs(phi - thick) > 1e-5
    assert far.sum() > 0.99 * len(pos)
    assert expect[far].any() and (expect[far] != (1 | 2 | 4)).any()
    assert np.array_equal(masks[far], expect[far])
    s.clear()
    assert s.colliderContacts().size == 0


# ---- 4. one free node against a float64 restatement of the PD substep -------------------------------------------
def np_pd_free_node(x0, cols, o, ticks):
    h = o.fixedTimestepSize / o.timeSubsteps
    m, x, v = 1.0, np.array(x0, np.float64), np.zeros(3)
    traj = []
    for _ in range(ticks):
        for _ in range(o.timeSubsteps):
            prev = x.copy()
            x = x + h * v
            msn = x * m / (h * h)
            mask = [k for k, c in enumerate(cols) if np_phi(c, x)[0][0] < o.collisionThickness]
            for _ in range(o.iterations):
                rhs = msn + sum(W * np_project(cols[k], x[None])[0] for k in mask) if mask else msn
                x = rhs / (m / (h * h) + W * len(mask))
            for k in mask:
                x = np_project(cols[k], x[None])[0]
            v = (1.0 - o.damping) * (x - prev) / h + np.array([0.0, -h * o.gravity, 0.0])
            for k in mask:
                n = np_phi(cols[k], x[None])[1][0]
                t = v - (v @ n) * n
                fr = 1.0 if np.linalg.norm(t) < o.staticFrictionThreshold else o.friction
                v = v - fr * t
        traj.append(x.copy())
    return np.array(traj)


@pytest.mark.parametrize("case", ["tilted_halfspace", "sphere", "box_edge"])
def test_free_node_matches_closed_form(pb, case):
    r45 = np.array([[np.cos(np.pi / 4), -np.sin(np.pi / 4), 0], [np.sin(np.pi / 4), np.cos(np.pi / 4), 0], [0, 0, 1]])
    cols, x0 = {
        "tilted_halfspace": ([pb.halfspace((0, 0, 0), (0.3, 1.0, 0.1))], (0.2, 2.0, -0.1)),
        "sphere": ([pb.sphere((0, 0, 0), 1.0), pb.halfspace((0, -1.5, 0), (0, 1, 0))], (0.3, 3.0, 0.2)),
        "box_edge": ([pb.box((0, 0, 0), (1, 1, 1), r45), pb.halfspace((0, -2.0, 0), (0, 1, 0))],
                     (0.05, np.sqrt(2.0) + 2.0, 0.3)),
    }[case]
    drop = x0[1]   # the height the node is dropped from
    s = pb.Solver(iterations=4)
    s.appendNodes(np.float32([x0]), radius=0.1, invMass=1.0)
    s.setColliders(cols)
    got = []
    for _ in range(100):
        s.tick()
        got.append(s.positions[0].astype(np.float64))
    assert not s.simFailed
    got = np.array(got)
    ref = np_pd_free_node(np.float32(x0).astype(np.float64), cols, s.getOptions(), 100)
    assert np.abs(got - ref).max() <= 1e-5 * drop, (case, np.abs(got - ref).max())
    assert (got[:, 1] < x0[1] - 0.5).any()   # it fell and met the collider


# ---- 5. fused and two-kernel paths agree with colliders, a bin keeps the stack --------------------------------------
BIN_SCRIPT = """import sys; sys.path.insert(0, %r)
import numpy as np
import pies_b200 as pb
from pies_b200 import scenes
s = pb.Solver(**scenes.S3_OPTIONS)
scenes.build_s3(s, bodies=48, nx=2, nz=2)
pos = s.positions
lo, hi = pos.min(0) - 0.5, pos.max(0) + 0.5
walls = [pb.halfspace((lo[0], 0, 0), (1, 0, 0)), pb.halfspace((hi[0], 0, 0), (-1, 0, 0)),
         pb.halfspace((0, 0, lo[2]), (0, 0, 1)), pb.halfspace((0, 0, hi[2]), (0, 0, -1))]
s.setColliders(walls)
body = np.arange(len(pos)) // 27
vel = np.zeros_like(pos)
vel[:, 0] = np.where(body %% 2 == 0, -3.0, 3.0)
vel[:, 2] = np.where((body // 2) %% 2 == 0, -2.0, 2.0)
s.setState(vel=vel.astype(np.float32))
P, V = [], []
for t in range(%d):
    s.tick()
    P.append(s.positions); V.append(s.velocities)
np.savez(sys.argv[1], pos0=pos, vel0=vel, pos=np.array(P), vel=np.array(V), prev=s.prevPositions, failed=np.array(s.simFailed),
         lo=lo, hi=hi, h=np.float32(s.getOptions().fixedTimestepSize / s.getOptions().timeSubsteps))
"""


def _bin_run(path, fused, ticks):
    env = dict(os.environ)
    env.pop("PIES_B200_NO_FUSED_LOCAL", None)
    if not fused:
        env["PIES_B200_NO_FUSED_LOCAL"] = "1"
    subprocess.run([sys.executable, "-c", BIN_SCRIPT % (ROOT, ticks), str(path)], check=True, env=env)
    return np.load(path)


def test_bin_fused_and_two_kernel_agree(pb, tmp_path):
    ticks = 60
    a = _bin_run(tmp_path / "fused.npz", True, ticks)
    b = _bin_run(tmp_path / "two_kernel.npz", False, ticks)
    for k in ("pos", "vel", "prev"):
        assert np.array_equal(a[k], b[k]), k
    assert not a["failed"] and np.isfinite(a["pos"]).all() and np.isfinite(a["vel"]).all()
    pos, vel, lo, hi, h = a["pos"], a["vel"], a["lo"], a["hi"], float(a["h"])
    phi = np.stack([pos[..., 0] - lo[0], hi[0] - pos[..., 0], pos[..., 2] - lo[2], hi[2] - pos[..., 2]], axis=-1)
    vmax = max(np.linalg.norm(vel, axis=-1).max(), np.linalg.norm(a["vel0"], axis=-1).max())
    assert phi.min() >= -h * vmax, (phi.min(), h * vmax)
    assert phi[-10:].min() >= -1e-4, phi[-10:].min()
    assert (phi[: ticks // 2].min(axis=(0, 2)) < 0.1).any()   # the bodies did reach the walls
    # kinetic energy (unit mass per node) never exceeds the initial kinetic plus potential energy above the floor
    ke = 0.5 * (vel ** 2).sum(axis=(1, 2))
    bound = 0.5 * (a["vel0"].astype(np.float64) ** 2).sum() + 10.0 * a["pos0"][:, 1].astype(np.float64).sum()
    assert ke.max() <= 1.05 * bound, (ke.max(), bound)


# ---- 6. PBD ------------------------------------------------------------------------------------------------------------
def test_pbd_bin_and_sphere(pb):
    from pies_b200 import scenes
    s = pb.Solver(solver="PBD")
    scenes.build_pbd_boxes(s)
    pos = s.positions
    cols = bin_walls(pos, 1.0, pb) + [pb.sphere((9.5, 1.0, 1.5), 1.0)]
    s.setColliders(cols)
    r = s.getVertices()["radius"].astype(np.float64)
    for _ in range(80):
        s.tick()
        p = s.positions
        assert np.isfinite(p).all()
        for c in cols:
            phi, _ = np_phi(c, p)
            assert (phi - r >= -1e-5).all()
    assert not s.simFailed


def test_pbd_friction_on_a_collider(pb):
    # free nodes resting on a collider plane (the floor is moved out of the way): the floor's rule in the collider's
    # tangent plane stops a slow node (planar speed < 5) and scales a fast one by 1 - friction
    s = pb.Solver(solver="PBD", floorHeight=-10.0)
    s.appendNodes(np.float32([[0, 0.1, 0], [5, 0.1, 0], [10, 0.1, 0]]), radius=0.1, invMass=1.0)
    s.setColliders([pb.halfspace((0, 0, 0), (0, 1, 0))])
    v0 = np.float32([[1.0, 0, 0.5], [0, 0, -2.0], [8.0, 0, 0]])
    s.setState(vel=v0)
    s.tick()
    o = s.getOptions()
    p, v = s.positions, s.velocities
    assert np.allclose(p[:, 1], 0.1, atol=1e-7)                     # clamped onto the plane
    assert np.array_equal(v[:2, [0, 2]], np.zeros((2, 2), np.float32))
    assert v[2, 0] == pytest.approx(8.0 * (1.0 - o.damping) * (1.0 - o.friction), rel=1e-4)
    assert v[2, 2] == 0.0


# ---- 7. argument checks ----------------------------------------------------------------------------------------------
def test_set_colliders_rejects_bad_sets(pb):
    s = pb.Solver()
    s.createTetBox((0, 1, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    ok = pb.sphere((0, 0, 0), 1.0)
    bad = []
    c = pb.Collider(kind=7); bad.append(c)                                           # unknown kind
    c = pb.sphere((0, np.nan, 0), 1.0); bad.append(c)                                # non-finite
    c = pb.box((0, 0, 0), (1, 1, 1)); c.axes[4] = np.inf; bad.append(c)
    bad.append(pb.halfspace((0, 0, 0), (0, 0, 0)))                                   # zero normal
    bad.append(pb.sphere((0, 0, 0), 0.0)); bad.append(pb.sphere((0, 0, 0), -1.0))   # radius <= 0
    bad.append(pb.box((0, 0, 0), (1, 0, 1)))                                         # half extent <= 0
    bad.append(pb.box((0, 0, 0), (1, 1, 1), [[1, 0, 0], [0, 1, 0.05], [0, 0, 1]]))   # not orthonormal
    bad.append(pb.box((0, 0, 0), (1, 1, 1), np.eye(3) * 1.001))
    for b in bad:
        with pytest.raises(pb.PiesError, match="error -1"):
            s.setColliders([ok, b])
    with pytest.raises(pb.PiesError, match="error -4"):
        s.setColliders([ok] * 33)
    s.setColliders([ok] * 32)
    # a rejected set leaves the previous one in place; clear() removes it
    s.setColliders([pb.halfspace((0, 1.5, 0), (0, 1, 0))])
    with pytest.raises(pb.PiesError):
        s.setColliders([pb.sphere((0, 0, 0), 0.0)])
    s.detect()
    assert s.colliderContacts().any()
    s.clear()
    s.createTetBox((0, 1, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    s.detect()
    assert not s.colliderContacts().any()
    # nearly orthonormal within 1e-4 is accepted
    e = 3e-5
    s.setColliders([pb.box((0, 0, 0), (1, 1, 1), [[1, e, 0], [-e, 1, 0], [0, 0, 1]])])
