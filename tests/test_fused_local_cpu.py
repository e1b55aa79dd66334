"""Closed segments of the fused local step + RHS (HostSystem::segs, `k_tet_rhs`) checked on the host without a GPU:
every segment is closed (its elements touch only its nodes, its nodes only its elements' tet slots), segments and the
residual lists cover every element and node exactly once, the segment-local gather list is the global one, and bodies
over the cap or with other constraint types stay on the two-kernel path."""
import numpy as np
import pytest

from pies_b200 import scenes, solver

TET_BOX, SHEET, SHAPE_BOX, MESH = 0, 1, 2, 3
SEG_ELEMS = SEG_NODES = 256


def tet_box(x, y=1.0):
    return [TET_BOX, x, y, 0.0, 1.0, 1000.0, 1.0, 0.0]


MIXED = [tet_box(0), tet_box(3), tet_box(6), [SHEET, 0.0, 6.0, 0.0, 1.0, 1.0, 1000.0, 0.0]] + \
        [tet_box(3 * i, 10.0) for i in range(7)] + [[SHAPE_BOX, 0.0, 20.0, 0.0, 3, 4, 4, 0.5]] + \
        [[MESH, 30.0, 3.07, 0.0, 0, 0, 0, 0], tet_box(40), tet_box(43)]


def _nodes_per_command(cmds, mesh):
    return [len(solver.probe_segments([c], *mesh)["incPtr"]) - 1 for c in cmds]


def _check_layout(g):
    inc_ptr, inc, slot, ids, base = g["incPtr"], g["inc"].astype(np.int64), g["segSlot"].astype(np.int64), g["elemIds"], g["baseTet"]
    n, ne = len(inc_ptr) - 1, len(ids)
    node_hits, elem_hits = np.zeros(n, int), np.zeros(ne, int)
    for n0, n1, e0, e1 in g["segs"].astype(np.int64):
        assert 0 < n1 - n0 <= SEG_NODES and 0 <= e1 - e0 <= SEG_ELEMS
        node_hits[n0:n1] += 1
        elem_hits[e0:e1] += 1
        assert ((ids[e0:e1] >= n0) & (ids[e0:e1] < n1)).all()                # elements reference only segment nodes
        rows = slice(inc_ptr[n0], inc_ptr[n1])
        assert ((inc[rows] >= base + 4 * e0) & (inc[rows] < base + 4 * e1)).all()   # nodes see only segment tet slots
        assert np.array_equal(base + 4 * e0 + slot[rows], inc[rows])           # local list == global list, row for row
    node_hits[g["restNodes"]] += 1
    elem_hits[g["restElems"]] += 1
    assert (node_hits == 1).all() and (elem_hits == 1).all()                  # everything exactly once
    assert (np.diff(g["restNodes"].astype(np.int64)) > 0).all() and (np.diff(g["restElems"].astype(np.int64)) > 0).all()


def test_s3_boxes_pack_five_bodies_per_segment():
    g = solver.probe_segments([tet_box(3 * i) for i in range(12)])
    _check_layout(g)
    assert len(g["restNodes"]) == 0 and len(g["restElems"]) == 0
    seg = g["segs"].astype(np.int64)
    assert (seg[:, 1] - seg[:, 0]).tolist() == [135, 135, 54]                # 5 + 5 + 2 bodies of 27 nodes
    assert (seg[:, 3] - seg[:, 2]).tolist() == [240, 240, 96]                # ... of 48 fused tets
    assert (seg[1:, 0] == seg[:-1, 1]).all() and (seg[1:, 2] == seg[:-1, 3]).all()


def test_mixed_scene_keeps_other_bodies_on_the_two_kernel_path():
    pts, tets, _ = scenes.cube24_mesh()
    mesh = (pts, tets)
    g = solver.probe_segments(MIXED, *mesh)
    _check_layout(g)
    counts = _nodes_per_command(MIXED, mesh)
    starts = np.concatenate([[0], np.cumsum(counts)])
    rest = set(g["restNodes"].tolist())
    covered_by_kind = {}
    for c, a, b in zip(MIXED, starts[:-1], starts[1:]):
        inside = [i not in rest for i in range(a, b)]
        covered_by_kind.setdefault(c[0], []).append(all(inside) if c[0] == TET_BOX else not any(inside))
    assert all(covered_by_kind[TET_BOX])                  # every tet box is in a segment
    assert all(covered_by_kind[SHEET])                    # distance constraints: residual
    assert all(covered_by_kind[SHAPE_BOX])                # shape matching: residual
    assert all(covered_by_kind[MESH])                     # TetGen cube of 16 546 tets: over the cap, residual
    assert len(g["restElems"]) == len(tets)               # its elements are the only residual tets
    seg = g["segs"].astype(np.int64)
    assert (seg[:, 1] - seg[:, 0]).tolist() == [81, 135, 54, 54]   # runs are cut by the bodies between them


def test_scene_without_tets_has_no_segments_with_elements():
    g = solver.probe_segments([[SHEET, 0.0, 1.0, 0.0, 1.0, 1.0, 1000.0, 0.0], [SHAPE_BOX, 0.0, 5.0, 0.0, 2, 2, 2, 0.5]])
    _check_layout(g)
    assert len(g["segs"]) == 0 and len(g["restNodes"]) == len(g["incPtr"]) - 1


def test_bad_command_is_rejected():
    with pytest.raises(solver.PiesError):
        solver.probe_segments([[7, 0, 0, 0, 0, 0, 0, 0]])
