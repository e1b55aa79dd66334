"""Whole-path parity (GPU, through the C ABI): scene construction, collision detection and
trajectories against golden data from the unmodified reference, plus size-independent properties."""
import numpy as np
import pytest

from conftest import bbox_diag, golden, noise_floor

pytestmark = pytest.mark.gpu

FACTORIES = {
    "tetbox": lambda s: s.createTetBox((0.25, 3.0, -1.5), 1.0, (0.5, 0.0, -0.25), 1000.0, 2.0, False),
    "tetbox_hinged": lambda s: s.createTetBox((0.0, 1.0, 0.0), 0.5, (0, 0, 0), 500.0, 1.0, True),
    "box": lambda s: s.createBox((1.0, 2.0, 3.0), 0.5, 100.0),
    "sheet": lambda s: s.createSheet((0.0, 5.0, 0.0), 0.25, 0.5, 200.0),
    "bendsheet": lambda s: s.createBendSheet((0.0, 4.0, 0.0), 0.5, 50.0),
    "shapebox": lambda s: s.createShapeMatchingBox((0.0, 2.0, 0.0), 3, 4, 5, 1.0, (0, 0, 0), 800.0),
    "shapesheet": lambda s: s.createShapeMatchingSheet((0.0, 6.0, 0.0), 0.2, (0, 0, 0), 300.0),
}


def two_box(s):
    s.createTetBox((0.1, 0.3, 0.1), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    s.createTetBox((0.4, 2.6, 0.3), 1.0, (0, -5, 0), 1000.0, 1.0, False)


@pytest.mark.parametrize("name", sorted(FACTORIES))
def test_factories_build_the_reference_scene(pb, name):
    """Node ids, positions, radii, triangles and lines are integer/byte work: bit-exact."""
    g = golden("factories")
    s = pb.Solver()
    FACTORIES[name](s)
    v = s.getVertices()
    assert (v["position"] == g[name + "_pos"]).all()
    assert (v["radius"] == g[name + "_radius"]).all()
    assert (s.velocities == g[name + "_vel"]).all()
    assert (s.getTriangles() == g[name + "_tris"].reshape(-1, 3)).all()
    assert (s.getLines() == g[name + "_lines"]).all()


@pytest.mark.parametrize("name", ["tetbox", "tetbox_hinged", "box", "sheet", "bendsheet", "shapebox"])
def test_factory_trajectories(pb, name):
    """10 PD ticks per primitive (default options): positions within 1e-4 x bbox diagonal of the reference."""
    g = golden("factories")
    s = pb.Solver()
    FACTORIES[name](s)
    tol = 1e-4 * bbox_diag(g[name + "_pos"])
    for k in range(10):
        s.tick()
        err = np.abs(s.getVertices()["position"] - g[name + "_traj"][k]).max()
        assert err <= tol, (name, k + 1, err, tol)
    verr = np.abs(s.velocities - g[name + "_vel10"]).max()
    assert verr <= 1e-4 * bbox_diag(g[name + "_pos"]) / 0.012, (name, verr)


def test_detection_lists_bit_exact_on_reference_states(pb):
    """Feed the reference's own states into the detection pass: the point-triangle list and the floor
    list must be identical as sequences (canonical order and multiplicity, SURVEY F7/F8)."""
    g = golden("collisions")
    s = pb.Solver(iterations=10)
    two_box(s)
    s.tick()  # builds the device topology
    for t in (3, 10, 14, 30):
        s.setState(g["t%d_pos" % t], g["t%d_prev" % t], None)
        s.detect()
        assert (s.triCollisions() == g["t%d_tri" % t]).all(), t
        assert (s.staticCollisions() == g["t%d_floor" % t]).all(), t
    assert len(g["t3_tri"]) == 120 and len(g["t14_floor"]) == 44  # SURVEY Appendix B anchors


def test_cell_occupancy_bit_exact(pb):
    g = golden("collisions")
    s = pb.Solver(iterations=10)
    two_box(s)
    s.tick()
    s.setState(g["occ_pos"], g["occ_prev"], None)
    s.detect()
    cells, counts, members = s.triOccupancy()
    assert (cells == g["occ_cells"]).all()
    assert (counts == g["occ_counts"]).all()
    assert (members == g["occ_members"]).all()


def test_two_box_collision_counts_and_trajectory(pb):
    """Appendix B scene end to end: contact counts tick by tick, positions at K = 1, 10, 40 within the north_star
    tolerance of 1e-4 x diagonal.  One caveat, measured on the reference itself (tests/golden/sensitivity.json,
    two_box_eps_sweep): perturbed by 1e-6 or 2e-6 before every tick it stays within 0.5 of that tolerance at K = 40, but
    from 4e-6 (a few ulps) on, 5 of 32 seeds catch a threshold contact differently and land 4.9x or 50x the tolerance
    away.  Our global step is a CG, not the reference's fp32 Cholesky, so our per-tick positions differ from the
    reference's by a few ulps too: K = 40 is held to 1e-4 x diagonal whenever our contact counts equal the reference's
    at every tick, and to the reference's own first excursion mode (10x) when a threshold contact has flipped."""
    g = golden("collisions")
    s = pb.Solver(iterations=10)
    two_box(s)
    tol = 1e-4 * bbox_diag(g["traj1_pos"])
    same_contacts = True
    for t in range(40):
        s.tick()
        st = s.stats()
        same = (st.triCollisions, st.staticCollisions) == tuple(g["counts"][t])
        if t < 16:
            assert same, t
        same_contacts = same_contacts and same
        if t + 1 in (1, 10, 40):
            err = np.abs(s.positions - g["traj%d_pos" % (t + 1)]).max()
            assert err <= (tol if same_contacts else 10 * tol), (t + 1, err, tol, same_contacts)


def test_tetgen_cube_on_floor(pb):
    """Config 1 at reduced size: TetGen cube (mesh taken from the reference's TetGen run) falling on the floor."""
    g = golden("tetgen_cube")
    s = pb.Solver()
    s.addTetMeshVolume(g["points"], g["tets"], g["faces"], (0, 0, 0), 1.0, 1000.0, 0.8, 1.0, 1000.0, 1.0, 1.0)
    tol = 1e-4 * bbox_diag(g["points"])
    for t in range(1, 61):
        s.tick()
        if t in (1, 10, 30, 60):
            st = s.stats()
            assert (st.triCollisions, st.staticCollisions) == tuple(g["ncoll%d" % t]), t
            err = np.abs(s.positions - g["pos%d" % t]).max()
            assert err <= tol, (t, err, tol)   # 1e-4 x diagonal at every check tick, floor contact included


def test_stack_trajectory_k_1_10_100(pb):
    """Reduced config 3 (16 stacked bodies, iterations=10).  K = 1, 10, 40 (free fall + floor contact): within
    1e-4 x diagonal and identical contact counts.  From tick 41 the bodies land on each other at 5 m/s with flat faces
    parallel: dozens of point-triangle pairs sit exactly at the detection threshold, and the reference perturbed by one
    ulp (1e-6) per tick catches a different set of them than the unperturbed reference (tests/golden/sensitivity.json:
    it differs from ITSELF by 1.2e-2 at tick 44 and 0.19 at tick 50).  So: as long as our per-tick contact counts equal
    the reference's, K = 44 is held to 1e-4 x diagonal; once a threshold contact has been caught by only one side it
    is held to twice the reference's own noise floor (the floor is a maximum over four seeds of a heavy-tailed
    quantity), and K = 100 to aggregate state."""
    from pies_b200 import scenes
    g = golden("stack16")
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=16, nx=2, nz=2)
    diag = bbox_diag(g["pos1"])
    same_contacts = True
    for t in range(1, 101):
        s.tick()
        st = s.stats()
        same_contacts = same_contacts and (st.triCollisions, st.staticCollisions) == tuple(g["counts"][t - 1])
        if t <= 40:
            assert same_contacts, t       # nothing is near a threshold before the first impact
        if t in (1, 10, 40, 44, 50, 100):
            p = s.positions
            err = np.abs(p - g["pos%d" % t]).max()
            if t <= 40 or (t == 44 and same_contacts):
                assert err <= 1e-4 * diag, (t, err)
            elif t in (44, 50):
                assert err <= max(1e-4 * diag, 2.0 * noise_floor("stack16", t)), (t, err)
                assert abs(st.triCollisions - g["ncoll%d" % t][0]) <= 0.15 * g["ncoll%d" % t][0] + 8
            else:
                assert np.isfinite(p).all() and p[:, 1].min() >= -1e-3
                assert abs(p[:, 1].mean() - g["pos100"][:, 1].mean()) <= 0.05 * diag
                assert 0.5 * g["ncoll100"][0] <= st.triCollisions <= 2.0 * g["ncoll100"][0]


def test_shape_and_goal_matching(pb):
    """Config 4 ingredients: shape-matching boxes, a goal region driven by updateFixedRegions, a linked region."""
    g = golden("clusters")
    s = pb.Solver(iterations=6)
    for k in range(3):
        s.createShapeMatchingBox((3.0 * k, 1.0 + 0.1 * k, 0.0), 3, 3, 3, 1.0, (0, 0, 0), 1000.0)
    s.addFixedRegions(g["region"].reshape(1, 16), 1000.0)
    s.addLinkedRegions(g["linked"].reshape(1, 16), 500.0)
    diag = bbox_diag(g["pos1"])
    for t in range(1, 21):
        s.updateFixedRegions(g["xforms"][t - 1].reshape(1, 16))
        s.tick()
        if t in (1, 10, 20):
            err = np.abs(s.positions - g["pos%d" % t]).max()
            assert err <= 1e-4 * diag, (t, err)


def test_run_to_run_bit_stable(pb):
    """No atomics on float data anywhere: two runs of a contact-rich scene are bit-identical."""
    from pies_b200 import scenes
    out = []
    for _ in range(2):
        s = pb.Solver(**scenes.S3_OPTIONS)
        scenes.build_s3(s, bodies=16, nx=2, nz=2)
        for _ in range(45):
            s.tick()
        out.append((s.positions.copy(), s.velocities.copy(), s.triCollisions().copy()))
    assert (out[0][0] == out[1][0]).all() and (out[0][1] == out[1][1]).all() and (out[0][2] == out[1][2]).all()


def pile(s, n=10):
    """Ten tet boxes dropped at 2 m/s with alternating lateral offsets: they topple, so contacts reach side faces and
    the contact clusters grow past 32 nodes (reference run: one 67-node cluster at tick 34, 168 nodes at tick 60)."""
    for i in range(n):
        s.createTetBox((0.35 * (i % 2), 0.55 + 1.25 * i, 0.3 * ((i // 2) % 2)), 1.0, (0.0, -2.0, 0.0), 1000.0, 1.0, False)


def test_ordered_sweep_executors_agree(pb):
    """The ordered stabilisation / friction sweeps have three executors (registers for clusters <= 32 nodes, one CTA
    from shared memory up to 1024 nodes, ticketed dataflow through L2 above): all replay the reference's sequential
    order per node, so forcing every cluster above 32 nodes through the global dataflow executor must give the same
    result (same operations in the same order; only fp contraction may differ between the kernels).  Both executors
    start from the same snapshot of a toppling pile and advance two ticks."""
    s = pb.Solver(iterations=10)
    pile(s)
    for _ in range(44):
        s.tick()
    snap = [s.positions.copy(), s.prevPositions.copy(), s.velocities.copy()]
    out = []
    for dataflow_only in (False, True):
        s.setState(*snap)
        s.setTuning(dataflowSweepsOnly=dataflow_only)
        for _ in range(2):
            s.tick()
        st = s.stats()
        assert st.triCollisions > 100
        mid, large = st.reserved & 0xffff, st.reserved >> 16
        assert (mid == 0 and large > 0) if dataflow_only else (mid > 0 and large == 0), (mid, large)
        out.append((s.positions.copy(), s.velocities.copy(), s.triCollisions().copy()))
    assert (out[0][2] == out[1][2]).all()
    diag = bbox_diag(out[0][0])
    assert np.abs(out[0][0] - out[1][0]).max() <= 1e-6 * diag
    assert np.abs(out[0][1] - out[1][1]).max() <= 1e-3


def test_free_fall_matches_closed_form(pb):
    """Size-independent property: before any contact a stack in free fall follows
    v_{n+1} = (1-d) v_n - h g exactly (gravity enters through the velocity update only, SURVEY F12)."""
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=64, nx=4, nz=4)
    y0 = s.positions[:, 1].copy()
    v, y = 0.0, 0.0
    for _ in range(8):
        s.tick()
        y += 0.012 * v
        v = (1 - 0.006) * v - 0.012 * 10.0
    # fp32 stiffness rows do not sum exactly to M/h^2, which acts like a position-proportional ghost force
    # (same in the reference): allow 5e-5 relative to the height
    assert (np.abs((s.positions[:, 1] - y0) - y) <= 5e-5 * np.maximum(1.0, y0)).all()
    assert np.abs(s.velocities[:, 1] - v).max() < 5e-3
    # lateral drift from the same ghost force: the compiled reference shows 4.7e-3 on this scene after 8 ticks
    assert np.abs(s.velocities[:, [0, 2]]).max() < 1e-2


def test_full_size_scene_properties(pb):
    """BASELINE size (S3, 1 000 032 tets): a few ticks stay finite, counts are the documented ones, the
    per-iteration projection count is 2 000 064 + live contacts, and nothing falls through the floor."""
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s)
    assert len(s.getVertices()) == 562518 and len(s.getTriangles()) == 1000032
    for _ in range(3):
        s.tick()
    st = s.stats()
    assert st.staticProjections == 2000064
    assert st.projectionsLastTick == 10 * (2000064 + st.triCollisions + st.staticCollisions)
    p = s.getVertices()["position"]
    assert np.isfinite(p).all() and p[:, 1].min() > 0.0 and not s.simFailed


def test_sim_failed_latch(pb):
    """Hang guard (Solver.cpp:751-755): > 1000 triangles in one cell latches simFailed; tick becomes a no-op."""
    s = pb.Solver()
    n = 1100
    rng = np.random.default_rng(0)
    pos = (rng.uniform(0.1, 0.9, size=(3 * n, 3)) + np.array([0, 5, 0])).astype(np.float32)
    s.appendNodes(pos, radius=0.05, invMass=1.0)
    s.appendTriangles(np.arange(3 * n, dtype=np.uint32).reshape(n, 3))
    s.tick()
    assert s.simFailed
    before = s.positions.copy()
    s.tick()
    assert (s.positions == before).all()


def test_empty_scene_and_clear(pb):
    s = pb.Solver()
    s.tick()
    assert len(s.getVertices()) == 0
    s.createTetBox((0, 3, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    s.tick()
    s.clear()
    assert len(s.getVertices()) == 0 and len(s.getTriangles()) == 0
    s.tick()
    s.createTetBox((0, 3, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    s.tick()
    assert np.isfinite(s.positions).all()


def test_clear_then_smaller_scene_reads_only_the_new_scene(pb):
    """tick -> clear -> create a SMALLER scene -> getVertices with no getVertices in between: the stale device state of
    the old scene must not be scattered into (and past the end of) the new vertex mirror, and the collision readback
    must refuse instead of copying the old scene's row pointers."""
    s = pb.Solver(iterations=10)
    for k in range(4):
        s.createTetBox((3.0 * k, 0.3, 0.0), 1.0, (0, 0, 0), 1000.0, 1.0, False)   # resting on the floor: floor contacts
    for _ in range(20):
        s.tick()
    assert s.stats().staticCollisions > 0
    s.clear()
    s.createBox((1.0, 2.0, 3.0), 0.5, 100.0)           # 8 nodes instead of 108
    g = golden("factories")
    v = s.getVertices()
    assert len(v) == len(g["box_pos"]) and (v["position"] == g["box_pos"]).all()
    assert s.stats().staticCollisions == 0 and s.stats().triCollisions == 0
    with pytest.raises(pb.PiesError):
        s.collisionCsr()
    s.tick()
    assert np.isfinite(s.positions).all() and len(s.positions) == len(g["box_pos"])


def test_bodies_added_between_ticks(pb, ref):
    """Hosts add bodies while the simulation runs; both sides must agree afterwards."""
    r = ref.RefSolver()
    s = pb.Solver()
    for x in (r, s):
        x.createTetBox((0, 3, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    for _ in range(3):
        r.tick(); s.tick()
    for x in (r, s):
        x.createTetBox((4, 3, 0), 1.0, (0, 1, 0), 1000.0, 1.0, False)
    for _ in range(5):
        r.tick(); s.tick()
    assert np.abs(s.positions - r.positions).max() <= 1e-4 * bbox_diag(r.positions)


def test_collision_csr_is_the_reference_collision_matrix(pb):
    """The collision terms the CG mat-vec streams (detect.cu, k_ccsr_fill) are exactly the matrix the reference adds to S
    for the same lists: oracle/port.py restates that assembly (pinned against the compiled reference's own S + C_t in the
    CPU suite); here the device CSR of the reference's contact states must reproduce it entry for entry."""
    from oracle import port
    g = golden("collisions")
    s = pb.Solver(iterations=10)
    two_box(s)
    s.tick()
    n = len(s.getVertices())
    for t in (3, 10, 14, 30):
        s.setState(g["t%d_pos" % t], g["t%d_prev" % t], None)
        s.detect()
        assert (s.triCollisions() == g["t%d_tri" % t]).all()
        ptr, col, val, diag = s.collisionCsr()
        wptr, wcol, wval, wdiag = port.collision_csr(n, g["t%d_tri" % t], g["t%d_floor" % t])
        assert (ptr == wptr).all() and (diag.astype(np.float64) == wdiag).all(), t
        for i in range(n):   # same entries per row (the device orders a row by (point, triangle index), the port by node ids)
            a, b = slice(ptr[i], ptr[i + 1]), slice(wptr[i], wptr[i + 1])
            assert sorted(zip(col[a].tolist(), val[a].astype(np.float64).tolist())) == sorted(zip(wcol[b].tolist(), wval[b].tolist())), (t, i)
        dense = np.diag(diag.astype(np.float64))
        for i in range(n):
            np.add.at(dense[i], col[ptr[i]:ptr[i + 1]], val[ptr[i]:ptr[i + 1]].astype(np.float64))
        assert np.array_equal(dense, port.collision_matrix(n, g["t%d_tri" % t], g["t%d_floor" % t])), t


# ---- global solve by islands (islands.cu) ---------------------------------------------------------------
def _stack(pb, **tuning):
    from pies_b200 import scenes
    s = pb.Solver(**scenes.S3_OPTIONS)
    scenes.build_s3(s, bodies=48, nx=2, nz=2)   # four columns of twelve bodies: islands of up to 324 nodes once stacked
    if tuning:
        s.setTuning(**tuning)
    return s


@pytest.mark.parametrize("tiers_off,label", [(0, "all tiers"), (1, "no warp tier"), (3, "CTA-512 and CTA-1024 only"),
                                              (7, "CTA-1024 only"), (14, "warp tier + grid-wide CG restricted to the other islands")])
def test_island_solves_agree_with_grid_wide_cg(pb, tiers_off, label):
    """The island-local PCG (one warp / one CTA per connected component of S + C_t) and the grid-wide CG solve the same
    systems to the same tolerance.  Their iterates differ by fp32 rounding (a few 1e-6 per tick, which the dynamics
    integrate: scripts/diag_islands.py measured 1e-5 x diagonal after 40 ticks of the 16-body stack, 3e-5 x here), so the
    trajectories are compared within the north_star's 1e-4 x diagonal for as long as both runs see the same contact counts; after the first threshold contact that
    only one of them catches the scene diverges like the reference diverges from itself
    (tests/golden/sensitivity.json).  Every tier is forced in turn so each kernel variant runs."""
    a = _stack(pb, islandSolves=False)
    b = _stack(pb, islandTiersOff=tiers_off, islandBigTier=True)
    diag = bbox_diag(a.positions)
    seen = np.zeros(4, np.int64)
    same_contacts, compared, contact_ticks = True, 0, 0
    for t in range(1, 47):
        a.tick(); b.tick()
        sa, sb = a.stats(), b.stats()
        same_contacts = same_contacts and (sa.triCollisions, sa.staticCollisions) == (sb.triCollisions, sb.staticCollisions)
        assert sa.islandsGlobal == 0 or sum(sa.islandsTier) == 0
        if tiers_off != 14:
            assert sb.islandsGlobal == 0, (label, t)         # nothing in this scene is too large for a CTA
        elif sb.triCollisions:
            assert sb.islandsGlobal > 0 and sb.islandsTier[0] > 0   # both kinds: the grid-wide CG runs on the left-over rows only
        assert sb.pcgCapHits == 0 and sa.pcgCapHits == 0
        seen += np.array(list(sb.islandsTier))
        assert np.isfinite(b.positions).all()
        if same_contacts:
            err = np.abs(a.positions - b.positions).max()
            assert err <= 1e-4 * diag, (label, t, err)
            compared = t
            contact_ticks += int(sb.triCollisions > 0)
    assert compared >= 41 and contact_ticks >= 1, (label, compared, contact_ticks)
    for tier in range(4):
        if tiers_off & (1 << tier):
            assert seen[tier] == 0, (label, tier)
    assert seen.sum() > 0 and sb.triCollisions > 0


def test_island_block_table_overflow_path(pb, monkeypatch, tmp_path):
    """Islands with more preconditioner blocks than a CTA tier's shared-memory table apply those blocks from global
    memory: same result."""
    a = _stack(pb)
    for _ in range(46):
        a.tick()
    monkeypatch.setenv("PIES_B200_ISLAND_MAXBLOCKS", "3")
    import subprocess, sys, os
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; import pies_b200 as pb; from pies_b200 import scenes\n"
            "s = pb.Solver(**scenes.S3_OPTIONS); scenes.build_s3(s, bodies=48, nx=2, nz=2)\n"
            "[s.tick() for _ in range(46)]\n"
            "np.save(sys.argv[1], s.positions)" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    out = str(tmp_path / "pies_island_overflow.npy")
    subprocess.run([sys.executable, "-c", code, out], check=True, env=dict(os.environ))  # the env hook is read once per process
    b = np.load(out)
    assert np.abs(a.positions - b).max() <= 1e-6 * bbox_diag(b)   # same arithmetic from another memory space


@pytest.mark.parametrize("switch", ["PIES_B200_NO_DENSE", "PIES_B200_NO_DENSE2", "PIES_B200_NO_DENSE,PIES_B200_NO_SMALL_CTA",
                                    "PIES_B200_NO_CELL_TABLE"])
def test_island_list_switches_agree(pb, switch, tmp_path):
    """The A/B switches (no dense-inverse list, no 128-thread list, radix-sorted cell table) route the same
    work through the other kernels; all of them solve to the same tolerance, so the trajectories agree like the
    island / grid-wide pair above (compared while the contact counts agree)."""
    import subprocess, sys, os
    ticks = 44
    a = _stack(pb)
    counts_a = []
    for _ in range(ticks):
        a.tick()
        st = a.stats()
        counts_a.append((st.triCollisions, st.staticCollisions))
    code = ("import sys; sys.path.insert(0, %r); import numpy as np; import pies_b200 as pb; from pies_b200 import scenes\n"
            "s = pb.Solver(**scenes.S3_OPTIONS); scenes.build_s3(s, bodies=48, nx=2, nz=2)\n"
            "c = []\n"
            "for _ in range(%d):\n"
            "    s.tick(); st = s.stats(); c.append((st.triCollisions, st.staticCollisions, st.pcgCapHits))\n"
            "np.savez(sys.argv[1], pos=s.positions, counts=np.array(c))" % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), ticks))
    out = str(tmp_path / "pies_island_switch.npz")
    env = dict(os.environ)
    for name in switch.split(","):
        env[name] = "1"
    subprocess.run([sys.executable, "-c", code, out], check=True, env=env)   # the env hooks are read once per process
    b = np.load(out)
    assert (b["counts"][:, 2] == 0).all()
    assert np.isfinite(b["pos"]).all()
    if switch == "PIES_B200_NO_CELL_TABLE":   # radix-sorted cell table instead of the direct one: the same lists, bit for bit
        assert [tuple(r[:2]) for r in b["counts"]] == counts_a
        assert np.array_equal(a.positions, b["pos"])
    elif [tuple(r[:2]) for r in b["counts"]] == counts_a:
        assert np.abs(a.positions - b["pos"]).max() <= 1e-4 * bbox_diag(b["pos"]), switch
    else:   # a threshold contact caught by one run only: the scene diverges like the reference does from itself
        first = next(i for i, r in enumerate(b["counts"]) if tuple(r[:2]) != counts_a[i])
        assert first >= 30, (switch, first)


def test_island_trace_and_lists(pb):
    """Diagnostics entry point: the per-island record of the last global solve (rows, rounds / iterations, SM clocks,
    matrix entries) for every list, read in a process that has PIES_B200_ISLAND_TRACE set.  On the 4 x 12 stack at tick 46
    the dense-inverse lists hold the stacked columns (refinement: a handful of rounds), the warp list the free bodies."""
    import subprocess, sys, os, json
    code = ("import sys, json; sys.path.insert(0, %r); import numpy as np; import pies_b200 as pb; from pies_b200 import scenes\n"
            "s = pb.Solver(**scenes.S3_OPTIONS); scenes.build_s3(s, bodies=48, nx=2, nz=2)\n"
            "[s.tick() for _ in range(46)]\n"
            "st = s.stats()\n"
            "out = {'tiers': list(st.islandsTier), 'inv': int(st.islandInverseFloats), 'lists': {}}\n"
            "for slot in range(7):\n"
            "    tr = s.debugIslandTrace(slot)\n"
            "    out['lists'][str(slot)] = tr.tolist()\n"
            "print(json.dumps(out))" % os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    env = dict(os.environ, PIES_B200_ISLAND_TRACE="1")
    res = subprocess.run([sys.executable, "-c", code], check=True, env=env, capture_output=True, text=True)
    out = json.loads(res.stdout.strip().splitlines()[-1])
    lists = {int(k): np.array(v, dtype=np.int64).reshape(-1, 4) for k, v in out["lists"].items()}
    n_islands = sum(len(v) for v in lists.values())
    assert n_islands == sum(out["tiers"]) and n_islands > 0
    assert len(lists[1]) + len(lists[4]) + len(lists[5]) + len(lists[6]) == out["tiers"][1]
    rows = sum(int(v[:, 0].sum()) for v in lists.values())
    assert rows == 48 * 27                                       # every node is in exactly one island
    dense = np.concatenate([lists[5], lists[6]])
    assert len(dense) > 0 and dense[:, 0].max() <= 192 and (lists[5][:, 0] <= 128).all()
    assert (dense[:, 1] >= 1).all() and (dense[:, 1] <= 8).all()   # refinement rounds, not CG iterations
    assert (lists[0][:, 0] <= 32).all()
    expected_inv = sum(int(m) * (int(m) + 1) // 2 for m in lists[0][:, 0]) + sum(int(m) ** 2 for m in dense[:, 0]) \
        + sum(14 * int(m) for k in (1, 2, 3, 4) for m in lists[k][:, 0])
    assert out["inv"] == expected_inv


def test_pcg_cap_is_loud(pb):
    """A solve that stops at pcgMaxIterations far from its tolerance is reported: counter, residual and an error code
    (the reference's Cholesky cannot fail this way, so silence would hide a wrong trajectory)."""
    s = _stack(pb, pcgMaxIterations=1, pcgTolerance=1e-12)
    # free fall is solved by one application of the exact block inverse (residual 1e-10 even at the cap); once the
    # bodies touch (tick ~30 on) one iteration per solve is far from enough
    with pytest.raises(pb.PiesError, match="not converged"):
        for _ in range(46):
            s.tick()
    st = s.stats()
    assert st.pcgCapHits > 0 and st.pcgWorstCapResidual > 1e-9


def test_svd_warm_start_matches_cold_start(pb):
    """k_tet_elems warm-starts the 3x3 Jacobi SVD of every tet from the rotations the previous PD iteration converged to
    (two quaternions per tet, state).  Any converged SVD gives the same projection U sigma^ V^T up to rounding, so the
    trajectory must follow the cold-started one: same contact counts, positions within the rounding-integration bound
    (3e-5 x diagonal over 40 ticks, cf. tests/golden/sensitivity.json) through free fall, rotation-free floor contact and
    — with a spinning, sheared body — large rotations between iterations."""
    from pies_b200 import scenes

    def make(warm):
        s = pb.Solver(**scenes.S3_OPTIONS)
        scenes.build_s3(s, bodies=16, nx=2, nz=2)
        s.createTetBox((9.0, 2.0, 0.0), 1.0, (0.0, 0.0, 0.0), 1000.0, 1.0, False)
        s.setTuning(svdWarmStart=warm)
        return s
    a, b = make(True), make(False)
    # spin and shear the extra body: node velocities v = omega x (r - c) + shear
    p = a.positions; n0 = 16 * 27
    c = p[n0:].mean(0)
    v = np.zeros_like(p)
    r = p[n0:] - c
    v[n0:] = np.cross(np.array([0.0, 0.0, 25.0], np.float32), r) + np.outer(r[:, 1], np.array([3.0, 0.0, 0.0], np.float32))
    for s in (a, b):
        s.setState(None, None, v)
    diag = bbox_diag(p)
    for t in range(1, 41):
        a.tick(); b.tick()
        sa, sb = a.stats(), b.stats()
        assert (sa.triCollisions, sa.staticCollisions) == (sb.triCollisions, sb.staticCollisions), t
        err = np.abs(a.positions - b.positions).max()
        assert err <= 3e-5 * diag, (t, err)
    assert np.isfinite(a.positions).all()


def test_device_vertex_array_and_external_render_buffer(pb):
    """Zero-copy readback: the Vertex array on the device (36 B per vertex, Solver.h:42-49) equals what getVertices()
    returns, both in the solver's own buffer and in a caller-supplied one (standing in for an imported Vulkan / OpenGL
    vertex buffer), with no host copy in between."""
    import torch
    s = pb.Solver(iterations=10)
    two_box(s)
    for _ in range(5):
        s.tick()
    ptr, n = s.deviceVertices()
    assert n == 54 and ptr

    class Raw:
        def __init__(self, p, n):
            self.__cuda_array_interface__ = {"shape": (n, 9), "typestr": "<f4", "data": (p, False), "version": 3, "strides": None}
    dev = torch.as_tensor(Raw(ptr, n), device="cuda").clone().cpu().numpy()
    host = s.getVertices()
    assert (dev[:, :3] == host["position"]).all() and (dev[:, 3] == host["radius"]).all()
    assert (dev[:, 4:7] == host["baseColor"]).all()
    ext = torch.zeros((n, 9), dtype=torch.float32, device="cuda")
    s.setVertexBuffer(ext.data_ptr())
    s.tick()
    p2, _ = s.deviceVertices()
    assert p2 == ext.data_ptr()
    torch.cuda.synchronize()
    host = s.getVertices()
    got = ext.cpu().numpy()
    assert (got[:, :3] == host["position"]).all() and (got[:, 3] == host["radius"]).all() and (got[:, 4:7] == host["baseColor"]).all()
    s.setVertexBuffer(None)
    s.tick()
    assert np.isfinite(s.getVertices()["position"]).all()
    with pytest.raises(pb.PiesError):
        s.setVertexBuffer(12345)
