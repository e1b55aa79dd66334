"""External forces and wind in the PD and PBD ticks (DESIGN.md section 11)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _wind_forces64(x, v, tris, w, cn, ct, host=None):
    """float64 restatement of f_i (include/pies_b200.h): per triangle f_t / 3 to each corner, plus the host force."""
    x = np.asarray(x, np.float64); v = np.asarray(v, np.float64)
    f = np.zeros_like(x) if host is None else np.asarray(host, np.float64).copy()
    ft_all = np.zeros((len(tris), 3))
    for t, (a, b, c) in enumerate(np.asarray(tris, np.int64)):
        m = np.cross(x[b] - x[a], x[c] - x[a])
        ln = np.linalg.norm(m)
        if ln == 0.0:
            continue
        n = m / ln
        u = (v[a] + v[b] + v[c]) / 3.0 - np.asarray(w, np.float64)
        un = u @ n
        ut = u - un * n
        ft = -(ln / 2.0) * (cn * un * abs(un) * n + ct * ut)
        ft_all[t] = ft
        for i in (a, b, c):
            f[i] += ft / 3.0
    return f, ft_all


def _triangle_scene(pb, solver, y=2.0, **opts):
    """One free horizontal right triangle of three unit-mass nodes (area 0.5), no constraints, floor far below."""
    s = pb.Solver(solver=solver, floorHeight=-1000.0, **opts)
    s.appendNodes(np.float32([[0, y, 0], [1, y, 0], [0, y, 1]]), radius=0.1, invMass=1.0)
    s.appendTriangles([[0, 1, 2]])
    return s


# ---- 1. no forces, same bits ------------------------------------------------------------------------------------------
def _no_force_states(pb, make, build, ticks):
    out = []
    for mode in ("never", "empty", "removed", "rejected", "cleared", "wind_removed"):
        s = make()
        build(s)
        n = len(s.positions)
        ids = np.array([0, n // 2], np.uint32)
        f = np.float32([[1.0, 2.0, 0.5], [-1.0, 0.0, 3.0]])
        if mode == "empty":
            s.setExternalForces([], np.zeros((0, 3)))
            s.setWind((0, 0, 0), 0.0, 0.0)
        elif mode == "removed":
            s.setExternalForces(ids, f)
            s.setExternalForces([], np.zeros((0, 3)))
        elif mode == "rejected":
            s.setExternalForces(ids, f)
            with pytest.raises(pb.PiesError):
                s.setExternalForces([n], f[:1])
            s.setExternalForces([], np.zeros((0, 3)))
        elif mode == "cleared":
            s.setExternalForces(ids, f)
            s.setWind((1.0, 2.0, 3.0), 1.0, 1.0)
            s.clear()
            build(s)
        elif mode == "wind_removed":
            s.setWind((1.0, 2.0, 3.0), 1.0, 1.0)
            s.setWind((1.0, 2.0, 3.0), 0.0, 0.0)
        for _ in range(ticks):
            s.tick()
        assert not s.simFailed
        assert not s.externalForces().any(), mode
        out.append((mode, s.positions, s.prevPositions, s.velocities))
        s.close()
    return out


@pytest.mark.parametrize("mode", ["pd_s3", "pbd"])
def test_no_forces_is_bit_identical(pb, mode):
    from pies_b200 import scenes
    if mode == "pd_s3":
        runs = _no_force_states(pb, lambda: pb.Solver(**scenes.S3_OPTIONS),
                                lambda s: scenes.build_s3(s, bodies=48, nx=2, nz=2), 48)
    else:
        runs = _no_force_states(pb, lambda: pb.Solver(solver="PBD"),
                                lambda s: s.createSheet((0.0, 2.0, 0.0), 0.5, 1.0, 0.8), 48)
    for m, *arrs in runs[1:]:
        for a, b in zip(runs[0][1:], arrs):
            assert np.isfinite(a).all()
            assert np.array_equal(a, b), m


# ---- 2. a free node under a constant host force against a float64 restatement ------------------------------------------
@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_free_node_host_force_matches_restatement(pb, solver):
    x0, F, im = np.float32([0.5, 1.5, -0.25]), np.float32([3.0, 6.0, -2.0]), 0.5
    s = pb.Solver(solver=solver, iterations=4, floorHeight=-100.0)
    s.appendNodes(x0[None], radius=0.1, invMass=im)
    s.setExternalForces([0], F[None])
    o = s.getOptions()
    h = o.fixedTimestepSize / o.timeSubsteps
    x, v = x0.astype(np.float64), np.zeros(3)
    Fd = F.astype(np.float64)
    grav = np.array([0.0, -o.gravity, 0.0])
    err = 0.0
    for _ in range(60):
        s.tick()
        for _ in range(o.timeSubsteps):
            prev = x.copy()
            if solver == "PD":   # the global solve of an unconstrained node returns its prediction
                x = x + h * v
                v = (1.0 - o.damping) * (x - prev) / h + h * grav + h * Fd * im
            else:
                x = x + v * h + grav * h * h + Fd * im * h * h
                v = (1.0 - o.damping) * (x - prev) / h
        err = max(err, np.abs(s.positions[0].astype(np.float64) - x).max())
    assert not s.simFailed
    disp = np.linalg.norm(x - x0)
    # PBD adds steps of order v h to positions of order 1, rounding each at ulp(x): its fp32 drift is ~30x PD's
    tol = (2e-5 if solver == "PD" else 3e-4) * disp
    assert err <= tol, (err, tol)
    assert np.allclose(s.externalForces()[0], F)
    # the force did act: the node went where gravity alone would not take it
    assert s.positions[0, 0] > x0[0] + 0.2 and s.positions[0, 1] > x0[1] - 0.5 * o.gravity * 0.72 ** 2 + 0.4


# ---- 3. wind forces at a given state ---------------------------------------------------------------------------------
def _sheet_state(s, seed):
    rng = np.random.default_rng(seed)
    p = s.positions
    pos = (p + rng.normal(scale=0.05, size=p.shape)).astype(np.float32)
    vel = rng.normal(size=p.shape).astype(np.float32)
    return pos, vel


@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_wind_forces_at_a_given_state(pb, solver):
    w, cn, ct = np.float32([1.5, -0.5, 2.0]), 0.8, 0.3
    s = pb.Solver(solver=solver, timeSubsteps=1)
    s.createSheet((0.0, 3.0, 0.0), 0.25, 0.5, 200.0 if solver == "PD" else 0.8)
    pos, vel = _sheet_state(s, 7)
    s.setState(pos=pos, prev=pos, vel=vel)
    hid = np.array([5, 17, 200], np.uint32)
    hf = np.float32([[1, 0, 0], [0, -2, 0.5], [0.25, 0.25, 0.25]])
    host = np.zeros_like(pos)
    host[hid] = hf
    s.setExternalForces(hid, hf)
    s.setWind(w, cn, ct)
    s.tick()
    got = s.externalForces().astype(np.float64)
    tris = s.getTriangles()
    ref, ft = _wind_forces64(pos, vel, tris, w, cn, ct, host)
    scale = np.abs(ref).max()
    assert scale > 0.1
    assert np.abs(got - ref).max() <= 1e-5 * scale, np.abs(got - ref).max() / scale
    # the triangles' forces and the host forces are all there is
    tot = ft.sum(0) + host.astype(np.float64).sum(0)
    assert np.abs(got.sum(0) - tot).max() <= 1e-5 * np.abs(got).sum(), (got.sum(0), tot)

    # reversing every triangle's winding on the same nodes gives the same forces
    def wind_only(tr):
        a = pb.Solver(solver=solver, timeSubsteps=1)
        a.appendNodes(pos, radius=0.125, invMass=2.0)
        a.appendTriangles(tr)
        a.setState(pos=pos, prev=pos, vel=vel)
        a.setWind(w, cn, ct)
        a.tick()
        return a.externalForces().astype(np.float64)
    f1, f2 = wind_only(tris), wind_only(tris[:, [0, 2, 1]])
    assert np.abs(f1 - f2).max() <= 1e-6 * np.abs(f1).max()
    assert np.abs(f1 + host - got).max() <= 1e-5 * scale


# ---- 4. terminal velocity --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_terminal_velocity(pb, solver):
    cn, area, im = 10.0, 0.5, 1.0
    s = _triangle_scene(pb, solver, y=2.0)
    s.setWind((0, 0, 0), cn, 0.0)
    o = s.getOptions()
    h, d, g = o.fixedTimestepSize / o.timeSubsteps, o.damping, o.gravity
    v, err = 0.0, 0.0
    for _ in range(200):
        s.tick()
        for _ in range(o.timeSubsteps):
            drag = -cn * area * v * abs(v) * im / 3.0
            if solver == "PD":
                v = (1.0 - d) * v + h * (-g + drag)
            else:
                v = (1.0 - d) * (v + h * (-g + drag))
        vy = s.velocities[:, 1].astype(np.float64)
        err = max(err, np.abs(vy - v).max())
    assert not s.simFailed
    vt = np.sqrt(3.0 * g / (cn * area * im))   # |v| where the drag balances gravity
    assert err <= 5e-4 * vt, err
    assert abs(v + vt) < 0.1 * vt                      # settled close to the terminal speed ...
    free = -g * h / d                                  # ... well below what damping alone allows in free fall
    assert abs(s.velocities[:, 1]).max() < 0.2 * abs(free)
    assert np.abs(s.velocities[:, [0, 2]]).max() <= 1e-6


# ---- 5. a pinned sheet in the wind -------------------------------------------------------------------------------------
def _sheet_under(pb, solver, wind, cn, ct):
    if solver == "PD":
        s = pb.Solver(iterations=10)
        s.createSheet((0.0, 4.0, 0.0), 0.25, 0.5, 200.0)
        ticks = 40
    else:   # the soft PBD sheet buckles among its touching nodes later on: look while the forces still dominate
        s = pb.Solver(solver="PBD")
        s.createSheet((0.0, 4.0, 0.0), 0.5, 1.0, 0.8)
        ticks = 10
    if cn or ct:
        s.setWind(wind, cn, ct)
    for _ in range(ticks):
        s.tick()
    assert not s.simFailed
    p = s.positions
    assert np.isfinite(p).all()
    return p


@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_pinned_sheet_in_wind(pb, solver):
    centre = 10 * 20 + 10
    u = 5.0 if solver == "PD" else 8.0   # per node, c_n A_i u^2 is about 0.6 (PD) and 3 (PBD) times its weight
    up = _sheet_under(pb, solver, (0, u, 0), 2.0, 0.0)[centre, 1]
    none = _sheet_under(pb, solver, (0, 0, 0), 0.0, 0.0)[centre, 1]
    down = _sheet_under(pb, solver, (0, -u, 0), 2.0, 0.0)[centre, 1]
    assert up > none > down, (up, none, down)
    xp = _sheet_under(pb, solver, (u, 0, 0), 2.0, 4.0)[:, 0].mean()
    x0 = _sheet_under(pb, solver, (0, 0, 0), 0.0, 0.0)[:, 0].mean()
    xm = _sheet_under(pb, solver, (-u, 0, 0), 2.0, 4.0)[:, 0].mean()
    assert xp > x0 > xm, (xp, x0, xm)


# ---- 6. launch counts --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_force_launch_counts(pb, solver):
    def launches(scene, host, wind):
        s = pb.Solver(solver=solver, iterations=4, timeSubsteps=2)
        if scene == "sheet":
            s.createSheet((0.0, 4.0, 0.0), 0.25, 0.5, 200.0 if solver == "PD" else 0.8)
        else:   # a rope: nodes and distance constraints, no triangles; its nodes never touch (PBD's node-node
            # pass launches differently when a pair comes within reach)
            s.appendNodes(np.float32([[1.0 * i, 4.0, 0.0] for i in range(10)]))
            s.appendDistanceConstraints([[i, i + 1] for i in range(9)], 100.0 if solver == "PD" else 0.8)
        if host:
            s.setExternalForces([1, 3], np.float32([[0.1, 0, 0], [0, 0.1, 0]]))
        if wind:
            s.setWind((0.1, 0.0, 0.0), 0.01, 0.01)
        s.tick()
        st = s.stats()
        assert not s.simFailed
        return st.kernelLaunchesLastTick, st.substepsLastTick
    for scene in ("sheet", "rope"):
        base, subs = launches(scene, False, False)
        assert subs == 2
        assert launches(scene, True, False)[0] == base, scene
        extra = 2 * subs if scene == "sheet" else 0
        assert launches(scene, False, True)[0] == base + extra, scene
        assert launches(scene, True, True)[0] == base + extra, scene


# ---- 7. lifetime ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_forces_persist_across_tick_n(pb, solver):
    def run(n_calls):
        s = _triangle_scene(pb, solver, y=5.0)
        s.appendNodes(np.float32([[4, 5, 0]]))
        s.setExternalForces([3], np.float32([[2, 1, 0]]))
        s.setWind((1, 0, 0.5), 1.0, 0.5)
        if n_calls == 1:
            s.tickN(5)
        else:
            for _ in range(5):
                s.tick()
        return s.positions, s.velocities, s.externalForces()
    a, b = run(1), run(5)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)
    assert np.array_equal(a[2][3], [2, 1, 0]) and np.abs(a[2][:3]).min() > 0


@pytest.mark.parametrize("solver", ["PD", "PBD"])
def test_forces_survive_appended_bodies(pb, solver):
    s = pb.Solver(solver=solver, floorHeight=-100.0)
    s.appendNodes(np.float32([[0, 5, 0]]))
    F = np.float32([3.0, 0.0, 0.0])
    s.setExternalForces([0], F[None])
    s.setWind((0, 0, 0), 1.0, 0.0)   # still air: only moving triangles feel it
    s.tick()
    assert np.array_equal(s.externalForces(), F[None])
    first = s.appendNodes(np.float32([[2, 5, 0], [3, 5, 0], [2, 5, 1]]), vel=np.float32([[0, -3, 0]] * 3))
    s.appendTriangles([[first, first + 1, first + 2]])
    f = s.externalForces()
    assert f.shape == (4, 3) and not f[1:].any()   # appended since the last tick
    vx = s.velocities[0, 0]
    s.tick()
    f = s.externalForces()
    assert np.array_equal(f[0], F)                      # the host force still acts on node 0 ...
    assert s.velocities[0, 0] > vx
    assert (f[1:, 1] > 0).all() and not f[1:, [0, 2]].any()   # ... the wind on the new triangle, against its fall
    assert not s.simFailed


# ---- 8. argument checks --------------------------------------------------------------------------------------------------
def test_force_and_wind_argument_checks(pb):
    import ctypes as C
    L = pb.lib()
    p = lambda a: a.ctypes.data_as(C.c_void_p)

    def make():
        s = _triangle_scene(pb, "PD", y=5.0)
        s.setState(vel=np.float32([[0, -2, 0]] * 3))
        return s
    a, b = make(), make()   # a sees every rejected call, b only the accepted ones
    F = np.float32([[1, 0, 0], [0, 0, 2]])
    for s in (a, b):
        s.setExternalForces([0, 2], F)
        s.setWind((0.5, 0, 0), 1.0, 0.5)
        s.tick()
    before = a.externalForces()
    assert np.array_equal(before, b.externalForces()) and before.any()
    n = len(a.positions)
    bad_forces = [([n - 1, n], F),                                   # id out of range
                  ([1, 1], F),                                       # duplicate
                  ([0, 1], np.float32([[np.nan, 0, 0], [0, 0, 0]])),
                  ([0, 1], np.float32([[0, 0, 0], [0, np.inf, 0]])),
                  ([0, 1], np.float32([[0, 0, 0], [0, 0, -np.inf]]))]
    for ids, f in bad_forces:
        with pytest.raises(pb.PiesError, match="error -1"):
            a.setExternalForces(ids, f)
        assert np.array_equal(a.externalForces(), before)
    bad_wind = [((np.nan, 0, 0), 1.0, 0.0), ((0, np.inf, 0), 1.0, 0.0), ((0, 0, 0), np.nan, 0.0),
                ((0, 0, 0), 1.0, np.inf), ((0, 0, 0), -1.0, 0.0), ((0, 0, 0), 1.0, -0.5)]
    for wv, cn, ct in bad_wind:
        with pytest.raises(pb.PiesError, match="error -1"):
            a.setWind(wv, cn, ct)
        assert np.array_equal(a.externalForces(), before)
    ids, f3, v3 = np.uint32([0]), np.float32([1, 2, 3]), np.float32([0, 0, 0])
    assert L.pies_b200_set_external_forces(a.h, 1, None, p(f3)) == -1
    assert L.pies_b200_set_external_forces(a.h, 1, p(ids), None) == -1
    assert L.pies_b200_set_wind(a.h, None, 1.0, 0.0) == -1
    assert L.pies_b200_get_external_forces(a.h, None) == -1
    # inside pd_tick_begin .. pd_tick_end
    a.pdTickBegin()
    assert L.pies_b200_set_external_forces(a.h, 1, p(ids), p(f3)) == -1
    assert L.pies_b200_set_external_forces(a.h, 0, None, None) == -1
    assert L.pies_b200_set_wind(a.h, p(v3), 0.0, 0.0) == -1
    a.pdSubstepBegin()
    for _ in range(a.getOptions().iterations):
        a.pdIteration()
    a.pdSubstepEnd(); a.pdTickEnd()
    b.tick()
    assert np.array_equal(a.externalForces(), b.externalForces())
    # the previous set and wind stayed in place through every rejection
    for _ in range(3):
        a.tick(); b.tick()
    for x, y in ((a.positions, b.positions), (a.velocities, b.velocities), (a.externalForces(), b.externalForces())):
        assert np.array_equal(x, y)
    assert L.pies_b200_set_external_forces(a.h, 0, None, None) == 0
    assert L.pies_b200_set_wind(a.h, p(v3), 0.0, 0.0) == 0
    a.tick()
    assert not a.externalForces().any()
