"""Drag targets in the PD and PBD ticks (DESIGN.md section 10)."""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _diag(p):
    return float(np.linalg.norm(p.max(0) - p.min(0)))


# ---- 1. no drag, same bits -----------------------------------------------------------------------------------------
def _no_drag_states(pb, make, build, ticks):
    out = []
    for mode in ("never", "empty", "removed", "rejected", "cleared"):
        s = make()
        build(s)
        n = len(s.positions)
        ids = np.array([0, n // 2], np.uint32)
        tgt = s.positions[ids] + np.float32([0.0, 2.0, 0.0])
        if mode == "empty":
            s.setDragTargets([], np.zeros((0, 3)), [])
        elif mode == "removed":
            s.setDragTargets(ids, tgt, [100.0, 100.0])
            s.setDragTargets([], np.zeros((0, 3)), [])
        elif mode == "rejected":
            s.setDragTargets(ids, tgt, [100.0, 100.0])
            with pytest.raises(pb.PiesError):
                s.setDragTargets([n], tgt[:1], [1.0])
            s.setDragTargets([], np.zeros((0, 3)), [])
        elif mode == "cleared":
            s.setDragTargets(ids, tgt, [100.0, 100.0])
            s.clear()
            build(s)
        for _ in range(ticks):
            s.tick()
        assert not s.simFailed
        out.append((mode, s.positions, s.prevPositions, s.velocities))
        s.close()
    return out


@pytest.mark.parametrize("mode", ["pd_s3", "pbd"])
def test_no_drag_is_bit_identical(pb, mode):
    from pies_b200 import scenes
    if mode == "pd_s3":
        runs = _no_drag_states(pb, lambda: pb.Solver(**scenes.S3_OPTIONS),
                               lambda s: scenes.build_s3(s, bodies=48, nx=2, nz=2), 48)
    else:
        runs = _no_drag_states(pb, lambda: pb.Solver(solver="PBD"),
                               lambda s: s.createSheet((0.0, 2.0, 0.0), 0.5, 1.0, 0.8), 48)
    for m, *arrs in runs[1:]:
        for a, b in zip(runs[0][1:], arrs):
            assert np.isfinite(a).all()
            assert np.array_equal(a, b), m


# ---- 2. a free node against a float64 restatement of the PD substep (no triangles: detection's early return) --------
def test_free_node_pd_matches_restatement(pb):
    # Near the origin with the floor moved far below: the fp32 rounding of msn = x / h^2 grows with |x|, and the
    # undamped swing towards the target carries it from tick to tick.
    x0, g, w = np.float32([0.5, -1.5, -0.25]), np.float32([1.5, 1.5, 0.75]), 100.0
    s = pb.Solver(iterations=4, floorHeight=-100.0)
    s.appendNodes(x0[None], radius=0.1, invMass=1.0)
    s.setDragTargets([0], g[None], [w])
    o = s.getOptions()
    h = o.fixedTimestepSize / o.timeSubsteps
    m, x, v = 1.0, x0.astype(np.float64), np.zeros(3)
    gd = g.astype(np.float64)
    err = 0.0
    for _ in range(60):
        s.tick()
        for _ in range(o.timeSubsteps):
            prev = x.copy()
            x = x + h * v
            msn = x * m / (h * h)
            for _ in range(o.iterations):
                x = (msn + w * gd) / (m / (h * h) + w)
            v = (1.0 - o.damping) * (x - prev) / h + np.array([0.0, -h * o.gravity, 0.0])
        err = max(err, np.abs(s.positions[0].astype(np.float64) - x).max())
    assert not s.simFailed
    assert err <= 1e-5 * np.linalg.norm(gd - x0), err
    assert np.linalg.norm(s.positions[0] - g) < 0.5 * np.linalg.norm(g - x0)   # it did move towards the target


# ---- 3. a drag equals a static position constraint at the same place ------------------------------------------------
def test_drag_equals_position_constraint(pb):
    def build(s):   # resting on the floor, each held by a node of its top layer
        for i in range(3):
            s.createTetBox((3.0 * i, 0.01, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    a, b = pb.Solver(iterations=10), pb.Solver(iterations=10)
    build(a); build(b)
    ids = np.array([6, 27 + 13, 54 + 26], np.uint32)
    w = 1000.0
    a.appendPositionConstraints(ids, w)
    b.setDragTargets(ids, b.positions[ids], np.full(3, w))
    for _ in range(60):
        a.tick(); b.tick()
    pa, pbb = a.positions, b.positions
    assert not a.simFailed and not b.simFailed
    assert len(a.staticCollisions()) > 0 and len(b.staticCollisions()) > 0   # floor contact
    assert np.abs(pa - pbb).max() <= 1e-4 * _diag(pa), np.abs(pa - pbb).max()


# ---- 4. every solve path sees the weight -----------------------------------------------------------------------------
def test_every_solve_path_sees_the_drag(pb):
    from pies_b200 import scenes

    def run(**tuning):
        s = pb.Solver(**scenes.S3_OPTIONS)
        scenes.build_s3(s, bodies=8, nx=2, nz=2)
        if tuning:
            s.setTuning(**tuning)
        for _ in range(20):   # the stack settles into contact
            s.tick()
        node = 13   # centre of the bottom body, below the one stacked on it
        s.setDragTargets([node], s.positions[node][None] + np.float32([0.3, 0.4, 0.0]), [5000.0])
        for _ in range(20):
            s.tick()
        assert not s.simFailed
        return s.positions
    ref = run()
    d = _diag(ref)
    for tuning in (dict(islandSolves=False), dict(islandTiersOff=1), dict(islandTiersOff=2), dict(islandTiersOff=4)):
        p = run(**tuning)
        assert np.abs(p - ref).max() <= 1e-4 * d, (tuning, np.abs(p - ref).max())


# ---- 5. fused and two-kernel paths stay bit-identical with drags, colliders and the floor ----------------------------
DRAG_SCRIPT = """import sys; sys.path.insert(0, %r)
import numpy as np
import pies_b200 as pb
from pies_b200 import scenes
s = pb.Solver(**scenes.S3_OPTIONS)
scenes.build_s3(s, bodies=48, nx=2, nz=2)
pos = s.positions
lo, hi = pos.min(0) - 0.5, pos.max(0) + 0.5
s.setColliders([pb.halfspace((lo[0], 0, 0), (1, 0, 0)), pb.halfspace((hi[0], 0, 0), (-1, 0, 0)), pb.sphere((0, -0.5, 0), 1.0)])
ids = np.arange(0, len(pos), 97, dtype=np.uint32)
P, V = [], []
for t in range(40):
    s.setDragTargets(ids, pos[ids] + np.float32([0.0, 0.05 * t, 0.0]), np.full(len(ids), 500.0))
    s.tick()
    P.append(s.positions); V.append(s.velocities)
np.savez(sys.argv[1], pos=np.array(P), vel=np.array(V), prev=s.prevPositions, failed=np.array(s.simFailed))
"""


def _drag_run(path, fused):
    env = dict(os.environ)
    env.pop("PIES_B200_NO_FUSED_LOCAL", None)
    if not fused:
        env["PIES_B200_NO_FUSED_LOCAL"] = "1"
    subprocess.run([sys.executable, "-c", DRAG_SCRIPT % ROOT, str(path)], check=True, env=env)
    return np.load(path)


def test_drag_fused_and_two_kernel_agree(pb, tmp_path):
    a = _drag_run(tmp_path / "fused.npz", True)
    b = _drag_run(tmp_path / "two_kernel.npz", False)
    assert not a["failed"] and np.isfinite(a["pos"]).all()
    for k in ("pos", "vel", "prev"):
        assert np.array_equal(a[k], b[k]), k


# ---- 6. launch counts --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("contact, extra", [("free_fall", 2), ("on_floor", 1)])
def test_drag_launch_counts(pb, contact, extra):
    # per substep, drags add k_drag_terms; a substep with no other one-node weight and no triangle contact also runs
    # k_ccsr_fill, which it otherwise skips
    y = 20.0 if contact == "free_fall" else 0.01

    def launches(drag):
        s = pb.Solver(iterations=4, timeSubsteps=2)
        for i in range(4):
            s.createTetBox((3.0 * i, y, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
        if drag is not None:
            s.setDragTargets([drag], s.positions[drag][None] + np.float32([0, 0.1, 0]), [10.0])
        s.tick()
        st = s.stats()
        assert not s.simFailed
        if contact == "on_floor":
            assert st.staticCollisions > 0
        return st.kernelLaunchesLastTick, st.substepsLastTick
    base, subs = launches(None)
    assert launches(None)[0] == base
    with_drag, _ = launches(40)
    assert with_drag - base == extra * subs, (with_drag, base, subs)


# ---- 7. a free node in PBD ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("w", [0.25, 3.0])
def test_free_node_pbd_matches_restatement(pb, w):
    x0, g = np.float32([0.5, 10.0, -0.25]), np.float32([1.5, 12.0, 0.75])
    s = pb.Solver(solver="PBD")
    s.appendNodes(x0[None], radius=0.1, invMass=1.0)
    s.setDragTargets([0], g[None], [w])
    o = s.getOptions()
    dt = o.fixedTimestepSize / o.timeSubsteps
    x, v = x0.astype(np.float64), np.zeros(3)
    gd = g.astype(np.float64)
    wc = min(w, 1.0)
    err = 0.0
    for _ in range(30):
        s.tick()
        for _ in range(o.timeSubsteps):
            prev = x.copy()
            x = x + dt * v + np.array([0.0, -o.gravity * dt * dt, 0.0])
            for _ in range(o.iterations):
                x = x + wc * (gd - x)
            v = (1.0 - o.damping) * (x - prev) / dt
        err = max(err, np.abs(s.positions[0].astype(np.float64) - x).max())
    assert not s.simFailed
    assert err <= 1e-5 * np.linalg.norm(gd - x0), err
    if w >= 1.0:   # a weight >= 1 puts the node on its target every iteration
        assert np.abs(s.positions[0] - g).max() <= 1e-5 * np.linalg.norm(gd - x0)


# ---- 8. interactive use: a box pulled up by one corner leaves the floor -------------------------------------------------
def test_dragged_box_lifts_off(pb):
    s = pb.Solver(iterations=10)
    s.createTetBox((0.0, 0.52, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    for _ in range(10):
        s.tick()
    p = s.positions
    c0 = p.mean(0)
    top = int(np.argmax(p[:, 1] + 1e-3 * p[:, 0] + 1e-6 * p[:, 2]))
    g = p[top].copy()
    for _ in range(80):
        g[1] += 0.03
        s.setDragTargets([top], g[None], [2.0e4])
        s.tick()
        assert np.isfinite(s.positions).all()
    assert not s.simFailed
    p = s.positions
    assert p.mean(0)[1] > c0[1] + 0.5
    assert p[:, 1].min() > 0.05   # off the floor


# ---- 10. argument checks ---------------------------------------------------------------------------------------------
def test_set_drag_targets_rejects_bad_sets(pb):
    import ctypes as C
    s = pb.Solver()
    s.createTetBox((0, 1, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    n = len(s.positions)
    g = np.float32([[0, 2, 0], [1, 2, 0]])
    bad = [([n - 1, n], g, [1.0, 1.0]),                       # id out of range
           ([3, 3], g, [1.0, 1.0]),                           # duplicate
           ([1, 2], np.float32([[0, np.nan, 0], [1, 2, 0]]), [1.0, 1.0]),
           ([1, 2], np.float32([[0, 2, 0], [np.inf, 2, 0]]), [1.0, 1.0]),
           ([1, 2], g, [1.0, np.inf]), ([1, 2], g, [np.nan, 1.0]),
           ([1, 2], g, [1.0, 0.0]), ([1, 2], g, [-1.0, 1.0])]  # weight <= 0
    for ids, tg, w in bad:
        with pytest.raises(pb.PiesError, match="error -1"):
            s.setDragTargets(ids, tg, w)
    L = pb.lib()
    ids = np.uint32([1]); tg = np.float32([0, 2, 0]); w = np.float32([1.0])
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    assert L.pies_b200_set_drag_targets(s.h, 1, None, p(tg), p(w)) == -1
    assert L.pies_b200_set_drag_targets(s.h, 1, p(ids), None, p(w)) == -1
    assert L.pies_b200_set_drag_targets(s.h, 1, p(ids), p(tg), None) == -1
    assert L.pies_b200_set_drag_targets(s.h, 0, None, None, None) == 0
    # inside pd_tick_begin .. pd_tick_end
    s.pdTickBegin()
    assert L.pies_b200_set_drag_targets(s.h, 1, p(ids), p(tg), p(w)) == -1
    s.pdSubstepBegin(); s.pdIteration(); s.pdSubstepEnd(); s.pdTickEnd()
    # a rejected set leaves the previous one in place: the node keeps being pulled up
    s.setDragTargets([1], np.float32([[0, 40, 0]]), [1.0e4])
    with pytest.raises(pb.PiesError):
        s.setDragTargets([1], np.float32([[0, 40, 0]]), [0.0])
    y0 = s.positions[1, 1]
    s.tick()
    assert s.positions[1, 1] > y0 + 0.1
    # appending a body keeps the set valid
    s.appendNodes(np.float32([[5, 5, 5]]))
    s.tick()
    assert s.positions[1, 1] > y0 + 0.2 and not s.simFailed
