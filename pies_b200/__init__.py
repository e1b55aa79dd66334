"""pies_b200 — B200-native implementation of the Pies per-timestep solver loop.

Python is only the test/bench harness here: the product is libpies_b200.so (CUDA, C ABI in
include/pies_b200.h) plus the header-only C++ drop-in Include/Pies/Solver.h.
"""
from .solver import (LIB_PATH, Collider, PiesError, Solver, SolverOptions, Stats, Tuning, VERTEX_DTYPE, box, halfspace,  # noqa: F401
                     lib, probe_ccd, probe_colliders, probe_edge_ccd, probe_node_range, probe_sort_pairs, probe_tet_projection, probe_tri_range,
                     probe_volume_projection, sphere)
