"""pies_b200_raycast against a float64 restatement of the documented Moller-Trumbore test (DESIGN.md section 10)."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def np_hits(o, d, P, tris):
    """float64: (t[R, T], u[R, T], v[R, T]) of every ray against every triangle, NaN where it is parallel or degenerate."""
    p0, p1, p2 = P[tris[:, 0]], P[tris[:, 1]], P[tris[:, 2]]
    e1, e2 = p1 - p0, p2 - p0
    pv = np.cross(d[:, None, :], e2[None])
    det = np.einsum("tk,rtk->rt", e1, pv)
    with np.errstate(divide="ignore", invalid="ignore"):
        inv = 1.0 / det
        sv = o[:, None, :] - p0[None]
        u = np.einsum("rtk,rtk->rt", sv, pv) * inv
        qv = np.cross(sv, e1[None])
        v = np.einsum("rk,rtk->rt", d, qv) * inv
        t = np.einsum("tk,rtk->rt", e2, qv) * inv
    bad = (det == 0) | (np.linalg.norm(np.cross(e1, e2), axis=1) == 0)[None]
    t[bad] = np.nan
    return t, u, v


def _deformed_boxes(pb):
    s = pb.Solver(iterations=10)
    for i in range(3):
        for j in range(2):
            s.createTetBox((2.5 * i + 0.3 * j, 0.6 + 2.6 * j, 0.2 * j), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    for _ in range(30):
        s.tick()
    assert not s.simFailed
    return s


def test_raycast_matches_float64(pb):
    s = _deformed_boxes(pb)
    P = s.positions.astype(np.float64)
    tris = np.array(s.getTriangles(), np.int64).reshape(-1, 3)
    rng = np.random.default_rng(11)
    nHit = 400
    f = rng.integers(0, len(tris), nHit)
    b = rng.uniform(0.05, 0.9, (nHit, 2))
    b[b.sum(1) > 0.95] *= 0.45
    tgt = P[tris[f, 0]] + b[:, :1] * (P[tris[f, 1]] - P[tris[f, 0]]) + b[:, 1:] * (P[tris[f, 2]] - P[tris[f, 0]])
    dirn = rng.normal(size=(nHit, 3))
    dirn /= np.linalg.norm(dirn, axis=1, keepdims=True)
    dist = rng.uniform(1.0, 6.0, nHit)
    o = tgt - dist[:, None] * dirn
    d = (tgt - o) * rng.uniform(0.5, 2.0, nHit)[:, None]   # not normalised
    # misses: straight up from above everything, and sideways far away
    top = P[:, 1].max() + 1.0
    om = np.concatenate([rng.uniform(-2, 8, (20, 3)) * [1, 0, 1] + [0, top, 0], rng.uniform(-2, 8, (20, 3)) + [0, 0, 50]])
    dm = np.concatenate([np.tile([0.0, 1.0, 0.0], (20, 1)), np.tile([1.0, 0.0, 0.0], (20, 1))])
    O = np.concatenate([o, om]).astype(np.float32)
    D = np.concatenate([d, dm]).astype(np.float32)
    tri, t, uv = s.raycast(O, D)
    T, U, V = np_hits(O.astype(np.float64), D.astype(np.float64), P, tris)
    lo = -1e-4
    cand = np.isfinite(T) & (T >= 0) & (U >= lo) & (V >= lo) & (U + V <= 1 - lo)
    Tc = np.where(cand, T, np.inf)
    best = np.argmin(Tc, axis=1)
    tb = Tc[np.arange(len(O)), best]
    srt = np.sort(Tc, axis=1)
    with np.errstate(invalid="ignore"):   # inf - inf on a miss: NaN, not robust
        gap = srt[:, 1] - srt[:, 0] if Tc.shape[1] > 1 else np.full(len(O), np.inf)
    ub, vb = U[np.arange(len(O)), best], V[np.arange(len(O)), best]
    robust = np.isfinite(tb) & (ub >= 1e-4) & (vb >= 1e-4) & (1 - ub - vb >= 1e-4) & (gap >= 1e-4)
    assert robust[:nHit].sum() > 0.8 * nHit
    r = robust
    assert np.array_equal(tri[r], best[r])
    assert np.allclose(t[r], tb[r], rtol=1e-5, atol=0)
    assert np.allclose(uv[r, 0], ub[r], atol=1e-5) and np.allclose(uv[r, 1], vb[r], atol=1e-5)
    # misses
    assert (tri[nHit:] == -1).all() and np.isinf(t[nHit:]).all() and (t[nHit:] > 0).all()
    assert (uv[nHit:] == 0).all()
    assert not np.isfinite(tb[nHit:]).any()
    # tMax cuts a hit; a tMax just past it keeps it
    rr = np.flatnonzero(r)[:50]
    tri2, t2, _ = s.raycast(O[rr], D[rr], (0.5 * tb[rr]).astype(np.float32))
    assert (tri2 == -1).all() and np.isinf(t2).all()
    tri3, t3, _ = s.raycast(O[rr], D[rr], (tb[rr] * (1 + 1e-3)).astype(np.float32))
    assert np.array_equal(tri3, tri[rr]) and np.array_equal(t3, t[rr])
    s.close()


def test_raycast_ties_go_to_the_lower_index(pb):
    s = pb.Solver()
    first = s.appendNodes(np.float32([[0, 1, 0], [2, 1, 0], [0, 1, 2], [0, 1, 0], [2, 1, 0], [0, 1, 2]]))
    ids = np.arange(first, first + 6, dtype=np.uint32)
    # triangle 0 and 2 share corners (2 reversed), triangle 1 uses copies of the same positions
    s.appendTriangles([[ids[0], ids[1], ids[2]], [ids[3], ids[4], ids[5]], [ids[0], ids[2], ids[1]]])
    o = np.float32([[0.5, 3.0, 0.5], [0.25, -2.0, 0.5]])
    d = np.float32([[0, -1, 0], [0, 2, 0]])   # from above and from below (two-sided)
    tri, t, uv = s.raycast(o, d)
    assert list(tri) == [0, 0]
    assert t[0] == np.float32(2.0) and t[1] == np.float32(1.5)
    assert np.allclose(uv, [[0.25, 0.25], [0.125, 0.25]], atol=1e-7)
    # set_state without a tick moves the hit
    p = s.positions
    s.setState(pos=p + np.float32([0, 0.5, 0]))
    tri, t, _ = s.raycast(o[:1], d[:1])
    assert tri[0] == 0 and t[0] == np.float32(1.5)


def test_raycast_without_triangles(pb):
    o, d = np.float32([[0, 5, 0]]), np.float32([[0, -1, 0]])
    s = pb.Solver()
    tri, t, uv = s.raycast(o, d)   # empty scene
    assert tri[0] == -1 and np.isinf(t[0]) and (uv == 0).all()
    s.appendNodes(np.float32([[0, 1, 0], [1, 1, 0], [0, 1, 1]]))
    tri, t, uv = s.raycast(o, d)   # nodes, no triangles
    assert tri[0] == -1 and np.isinf(t[0])
    tri, t, uv = s.raycast(np.zeros((0, 3)), np.zeros((0, 3)))
    assert len(tri) == 0


def test_raycast_rejects_bad_rays(pb):
    s = pb.Solver()
    s.createTetBox((0, 1, 0), 1.0, (0, 0, 0), 1000.0, 1.0, False)
    o, d = np.float32([[0.5, 5, 0.5]]), np.float32([[0, -1, 0]])
    for oo, dd, tm in ((np.float32([[np.nan, 5, 0]]), d, np.inf), (np.float32([[0, np.inf, 0]]), d, np.inf),
                       (o, np.float32([[0, 0, 0]]), np.inf), (o, np.float32([[0, np.nan, 0]]), np.inf),
                       (o, np.float32([[np.inf, -1, 0]]), np.inf), (o, d, np.nan), (o, d, -1.0)):
        with pytest.raises(pb.PiesError, match="error -1"):
            s.raycast(oo, dd, tm)
    tri, t, uv = s.raycast(o, d, np.inf)
    assert tri[0] >= 0 and t[0] == pytest.approx(2.0, abs=1e-5)
    tri, t, uv = s.raycast(o, d, 0.0)
    assert tri[0] == -1
    L = pb.lib()
    buf = [np.zeros(3, np.float32), np.float32([0, -1, 0]), np.float32([np.inf]), np.zeros(1, np.int32), np.zeros(1, np.float32),
           np.zeros(2, np.float32)]
    ptrs = [a.ctypes.data_as(C.c_void_p) for a in buf]
    for k in range(6):
        args = list(ptrs)
        args[k] = None
        assert L.pies_b200_raycast(s.h, 1, *args) == -1, k
    assert L.pies_b200_raycast(s.h, 0, None, None, None, None, None, None) == 0
