"""ctypes mirror of the reference's host API (Pies::Solver, reference Include/Pies/Solver.h:40-199)
over the C ABI of libpies_b200.so (include/pies_b200.h).

Method names, argument order and defaults follow the reference so parity tests read
like reference host code.  There is no CPU fallback: if the CUDA library is missing,
importing the binding raises; if no sm_100 device is present, Solver() raises.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpies_b200.so")

_f32p = np.ctypeslib.ndpointer(dtype=np.float32, flags="C_CONTIGUOUS")
_u32p = np.ctypeslib.ndpointer(dtype=np.uint32, flags="C_CONTIGUOUS")
_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_i64p = np.ctypeslib.ndpointer(dtype=np.int64, flags="C_CONTIGUOUS")
_u64p = np.ctypeslib.ndpointer(dtype=np.uint64, flags="C_CONTIGUOUS")


class SolverOptions(C.Structure):
    """Pies::SolverOptions (reference Include/Pies/Solver.h:23-38)."""
    _fields_ = [
        ("fixedTimestepSize", C.c_float), ("timeSubsteps", C.c_uint32),
        ("iterations", C.c_uint32), ("collisionStabilizationIterations", C.c_uint32),
        ("collisionThresholdDistance", C.c_float), ("collisionThickness", C.c_float),
        ("gravity", C.c_float), ("damping", C.c_float), ("friction", C.c_float),
        ("staticFrictionThreshold", C.c_float), ("floorHeight", C.c_float),
        ("gridSpacing", C.c_float), ("threadCount", C.c_uint32), ("solver", C.c_uint32),
    ]


class Tuning(C.Structure):
    _fields_ = [("pcgTolerance", C.c_float), ("pcgMaxIterations", C.c_uint32),
                ("pcgCheckEvery", C.c_uint32), ("reserved", C.c_uint32)]


class Stats(C.Structure):
    _fields_ = [
        ("staticProjections", C.c_uint64), ("collisionProjections", C.c_uint64),
        ("projectionsLastTick", C.c_uint64), ("pcgIterationsLastTick", C.c_uint64),
        ("kernelLaunchesLastTick", C.c_uint64),
        ("triCollisions", C.c_uint32), ("staticCollisions", C.c_uint32),
        ("substepsLastTick", C.c_uint32), ("simFailed", C.c_uint32),
        ("msTick", C.c_float), ("msLocal", C.c_float), ("msGlobal", C.c_float),
        ("msDetect", C.c_float), ("msContact", C.c_float), ("msOther", C.c_float),
        ("pcgLastRelResidual", C.c_float), ("msTetKernel", C.c_float),
        ("tetKernelLaunches", C.c_uint32), ("reserved", C.c_uint32),
        ("msSpmvKernel", C.c_float), ("msUpdateKernel", C.c_float), ("msGatherKernel", C.c_float),
        ("spmvKernelLaunches", C.c_uint32), ("updateKernelLaunches", C.c_uint32), ("gatherKernelLaunches", C.c_uint32),
        ("islandsTier", C.c_uint32 * 4), ("islandsGlobal", C.c_uint32), ("islandNodesGlobal", C.c_uint32),
        ("pcgCapHits", C.c_uint32), ("pcgWorstCapResidual", C.c_float),
        ("msIslandKernels", C.c_float), ("islandKernelLaunches", C.c_uint32),
        ("pcgIslandRowIterations", C.c_uint64),
        ("haloBytesLastTick", C.c_uint64), ("haloExchangesLastTick", C.c_uint32), ("msHalo", C.c_float),
        ("systemNonZeros", C.c_uint64), ("staticBodies", C.c_uint32), ("islandInverseFloats", C.c_uint32),
    ]


COLLIDER_HALFSPACE, COLLIDER_SPHERE, COLLIDER_BOX = 0, 1, 2
MAX_COLLIDERS = 32  # the width of the per-node contact mask


class Collider(C.Structure):
    """PiesB200Collider (include/pies_b200.h), 64 bytes: a static half-space, sphere or oriented solid box."""
    _fields_ = [("kind", C.c_uint32), ("center", C.c_float * 3), ("axes", C.c_float * 9), ("extent", C.c_float * 3)]


def halfspace(point, normal):
    """The half-space below the plane through `point` with outward `normal` (normalised here and again by the library)."""
    n = np.asarray(normal, np.float64).reshape(3)
    length = float(np.linalg.norm(n))
    if length > 0.0:
        n = n / length
    c = Collider(kind=COLLIDER_HALFSPACE)
    c.center[:] = [float(x) for x in np.asarray(point, np.float64).reshape(3)]
    c.axes[:] = [float(x) for x in n] + [0.0] * 6
    return c


def sphere(center, radius):
    c = Collider(kind=COLLIDER_SPHERE)
    c.center[:] = [float(x) for x in np.asarray(center, np.float64).reshape(3)]
    c.extent[:] = [float(radius), 0.0, 0.0]
    return c


def box(center, half_extents, axes=None):
    """Solid box; axes: 3 x 3 whose COLUMNS are the box's orthonormal local axes (default: the world axes)."""
    a = np.eye(3) if axes is None else np.asarray(axes, np.float64).reshape(3, 3)
    c = Collider(kind=COLLIDER_BOX)
    c.center[:] = [float(x) for x in np.asarray(center, np.float64).reshape(3)]
    c.axes[:] = [float(x) for x in a.T.reshape(9)]   # column after column
    c.extent[:] = [float(x) for x in np.asarray(half_extents, np.float64).reshape(3)]
    return c


def _collider_array(colliders):
    arr = (Collider * max(1, len(colliders)))()
    for i, c in enumerate(colliders):
        arr[i] = c
    return arr


VERTEX_DTYPE = np.dtype([("position", np.float32, 3), ("radius", np.float32),
                         ("baseColor", np.float32, 3), ("roughness", np.float32),
                         ("metallic", np.float32)])  # Solver::Vertex, 36 bytes

# every symbol include/pies_b200.h declares: name -> (restype, argtypes)
_vp = C.c_void_p
_SIGNATURES = {
    "pies_b200_default_options": (None, [C.POINTER(SolverOptions)]),
    "pies_b200_default_tuning": (None, [C.POINTER(Tuning)]),
    "pies_b200_create": (C.c_int, [C.POINTER(SolverOptions), C.c_int, C.POINTER(_vp)]),
    "pies_b200_destroy": (None, [_vp]),
    "pies_b200_last_error": (C.c_char_p, [_vp]),
    "pies_b200_set_tuning": (C.c_int, [_vp, C.POINTER(Tuning)]),
    "pies_b200_set_stream": (C.c_int, [_vp, _vp]),
    "pies_b200_get_options": (C.c_int, [_vp, C.POINTER(SolverOptions)]),
    "pies_b200_tick": (C.c_int, [_vp, C.c_float]),
    "pies_b200_tick_pd": (C.c_int, [_vp, C.c_float]),
    "pies_b200_tick_pbd": (C.c_int, [_vp, C.c_float]),
    "pies_b200_tick_n": (C.c_int, [_vp, C.c_uint32]),
    "pies_b200_set_release_hinge": (C.c_int, [_vp, C.c_int]),
    "pies_b200_get_render_state_dirty": (C.c_int, [_vp]),
    "pies_b200_set_render_state_dirty": (C.c_int, [_vp, C.c_int]),
    "pies_b200_sim_failed": (C.c_int, [_vp]),
    "pies_b200_clear": (C.c_int, [_vp]),
    "pies_b200_vertex_count": (C.c_uint32, [_vp]),
    "pies_b200_line_index_count": (C.c_uint32, [_vp]),
    "pies_b200_triangle_count": (C.c_uint32, [_vp]),
    "pies_b200_get_vertices": (_vp, [_vp]),
    "pies_b200_get_lines": (_vp, [_vp]),
    "pies_b200_get_triangles": (_vp, [_vp]),
    "pies_b200_add_nodes": (C.c_int, [_vp, C.c_uint32, _f32p]),
    "pies_b200_create_box": (C.c_int, [_vp, _f32p, C.c_float, C.c_float]),
    "pies_b200_create_tet_box": (C.c_int, [_vp, _f32p, C.c_float, _f32p, C.c_float, C.c_float, C.c_int]),
    "pies_b200_create_sheet": (C.c_int, [_vp, _f32p, C.c_float, C.c_float, C.c_float]),
    "pies_b200_create_shape_matching_box": (C.c_int, [_vp, _f32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, _f32p, C.c_float]),
    "pies_b200_create_shape_matching_sheet": (C.c_int, [_vp, _f32p, C.c_float, _f32p, C.c_float]),
    "pies_b200_create_bend_sheet": (C.c_int, [_vp, _f32p, C.c_float, C.c_float]),
    "pies_b200_add_tet_mesh_volume": (C.c_int, [_vp, C.c_uint32, _f32p, C.c_uint32, _u32p, C.c_uint32, _u32p, _f32p] + [C.c_float] * 7),
    "pies_b200_add_fixed_regions": (C.c_int, [_vp, C.c_uint32, _f32p, C.c_float]),
    "pies_b200_update_fixed_regions": (C.c_int, [_vp, C.c_uint32, _f32p]),
    "pies_b200_add_linked_regions": (C.c_int, [_vp, C.c_uint32, _f32p, C.c_float]),
    "pies_b200_append_nodes": (C.c_int, [_vp, C.c_uint32, _f32p, _f32p, _f32p, _f32p, C.POINTER(C.c_uint32)]),
    "pies_b200_append_distance_constraints": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float]),
    "pies_b200_append_position_constraints": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float]),
    "pies_b200_append_tet_constraints": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float, C.c_float, C.c_float]),
    "pies_b200_append_volume_constraints": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float, C.c_float, C.c_float]),
    "pies_b200_append_bend_constraints": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float]),
    "pies_b200_append_shape_constraint": (C.c_int, [_vp, C.c_uint32, _u32p, C.c_float]),
    "pies_b200_append_triangles": (C.c_int, [_vp, C.c_uint32, _u32p]),
    "pies_b200_get_positions": (C.c_int, [_vp, _f32p]),
    "pies_b200_get_prev_positions": (C.c_int, [_vp, _f32p]),
    "pies_b200_get_velocities": (C.c_int, [_vp, _f32p]),
    "pies_b200_set_state": (C.c_int, [_vp, _vp, _vp, _vp]),
    "pies_b200_detect": (C.c_int, [_vp]),
    "pies_b200_tri_collision_count": (C.c_uint32, [_vp]),
    "pies_b200_static_collision_count": (C.c_uint32, [_vp]),
    "pies_b200_get_tri_collisions": (C.c_int, [_vp, _u32p]),
    "pies_b200_get_collision_csr": (C.c_int, [_vp, C.POINTER(C.c_uint64), _vp, _vp, _vp, _vp]),
    "pies_b200_get_static_collisions": (C.c_int, [_vp, _u32p]),
    "pies_b200_tri_occupancy_counts": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "pies_b200_get_tri_occupancy": (C.c_int, [_vp, _i64p, _u32p, _u32p]),
    "pies_b200_detect_nodes": (C.c_int, [_vp]),
    "pies_b200_pd_tick_begin": (C.c_int, [_vp]),
    "pies_b200_pd_substep_begin": (C.c_int, [_vp]),
    "pies_b200_pd_iteration": (C.c_int, [_vp]),
    "pies_b200_pd_substep_end": (C.c_int, [_vp]),
    "pies_b200_pd_tick_end": (C.c_int, [_vp]),
    "pies_b200_device_state": (C.c_int, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]),
    "pies_b200_set_triangle_order": (C.c_int, [_vp, C.c_uint32, _u32p]),
    "pies_b200_set_owned_nodes": (C.c_int, [_vp, C.c_uint32, np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")]),
    "pies_b200_count_owned_contacts": (C.c_int, [_vp, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "pies_b200_set_vertex_buffer": (C.c_int, [_vp, _vp]),
    "pies_b200_device_vertices": (C.c_int, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_uint32)]),
    "pies_b200_halo_unique_id": (C.c_int, [_vp]),
    "pies_b200_halo_init": (C.c_int, [_vp, C.c_int, C.c_int, _vp]),
    "pies_b200_halo_set_lists": (C.c_int, [_vp, C.c_int, _vp, _vp, _vp, _vp, _vp]),
    "pies_b200_halo_exchange": (C.c_int, [_vp, C.c_int]),
    "pies_b200_halo_destroy": (C.c_int, [_vp]),
    "pies_b200_node_occupancy_counts": (C.c_int, [_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "pies_b200_get_node_occupancy": (C.c_int, [_vp, _i64p, _u32p, _u32p]),
    "pies_b200_get_stats": (C.c_int, [_vp, C.POINTER(Stats)]),
    "pies_b200_probe_tet_projection": (C.c_int, [C.c_uint32, _f32p, _f32p, C.c_float, C.c_float, _f32p]),
    "pies_b200_probe_volume_projection": (C.c_int, [C.c_uint32, _f32p, _f32p, C.c_float, C.c_float, _f32p]),
    "pies_b200_probe_ccd": (C.c_int, [C.c_uint32, _f32p, C.c_float, _i32p, _f32p]),
    "pies_b200_probe_edge_ccd": (C.c_int, [C.c_uint32, _f32p, _i32p, _f32p]),
    "pies_b200_debug_island_trace": (C.c_int, [_vp, C.c_int, _vp, C.c_uint32, C.POINTER(C.c_uint32)]),
    "pies_b200_probe_tri_range": (C.c_int, [C.c_uint32, _f32p, _f32p, _i64p, _u32p]),
    "pies_b200_probe_node_range": (C.c_int, [C.c_uint32, _f32p, _f32p, C.c_float, _i64p, _u32p]),
    "pies_b200_probe_sort_pairs": (C.c_int, [C.c_uint64, _u64p, _u32p, C.c_int]),
    "pies_b200_probe_sell": (C.c_int, [C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, C.POINTER(C.c_uint64)]),
    "pies_b200_set_colliders": (C.c_int, [_vp, C.c_uint32, _vp]),
    "pies_b200_get_collider_contacts": (C.c_int, [_vp, _u32p]),
    "pies_b200_probe_colliders": (C.c_int, [C.c_uint32, _vp, C.c_uint32, _vp, _vp, _vp]),
    "pies_b200_set_drag_targets": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp]),
    "pies_b200_raycast": (C.c_int, [_vp, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pies_b200_set_external_forces": (C.c_int, [_vp, C.c_uint32, _vp, _vp]),
    "pies_b200_set_wind": (C.c_int, [_vp, _vp, C.c_float, C.c_float]),
    "pies_b200_get_external_forces": (C.c_int, [_vp, _vp]),
    "pies_b200_probe_segments": (C.c_int, [C.c_uint32, _vp, C.c_uint32, _vp, C.c_uint32, _vp, _u64p] + [_vp] * 7),
}

_lib = None


def lib():
    """Loads libpies_b200.so; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError("%s not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
                              "or `make -C pies_b200/csrc` (no CPU fallback exists)" % LIB_PATH)
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


class PiesError(RuntimeError):
    pass


def _v3(v):
    return np.ascontiguousarray(np.asarray(v, dtype=np.float32).reshape(3))


class Solver:
    """Drop-in mirror of Pies::Solver.  `Solver(iterations=10, solver="PD")` == Solver(SolverOptions{...})."""

    def __init__(self, options=None, device=-1, **opts):
        L = lib()
        o = SolverOptions()
        L.pies_b200_default_options(C.byref(o))
        if options is not None:
            C.memmove(C.byref(o), C.byref(options), C.sizeof(o))
        for k, v in opts.items():
            if k == "solver":
                v = {"PBD": 0, "PD": 1}.get(v, v)
            if not hasattr(o, k):
                raise AttributeError(k)
            setattr(o, k, v)
        h = _vp()
        rc = L.pies_b200_create(C.byref(o), device, C.byref(h))
        if rc != 0:
            raise PiesError("pies_b200_create failed (%d): %s" % (rc, L.pies_b200_last_error(None).decode()))
        self.h = h
        self._options = o

    # -- plumbing --
    def _ck(self, rc):
        if rc != 0:
            raise PiesError("pies_b200 error %d: %s" % (rc, lib().pies_b200_last_error(self.h).decode()))

    def close(self):
        if getattr(self, "h", None):
            lib().pies_b200_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def setTuning(self, pcgTolerance=None, pcgMaxIterations=None, pcgCheckEvery=None, profilePhases=None, dataflowSweepsOnly=None,
                  islandSolves=None, islandTiersOff=None, islandBigTier=None, svdWarmStart=None, pbdColourBatches=None):
        t = Tuning()
        lib().pies_b200_default_tuning(C.byref(t))
        cur = getattr(self, "_tuning", None)
        if cur is not None:
            t = cur
        if pcgTolerance is not None: t.pcgTolerance = pcgTolerance
        if pcgMaxIterations is not None: t.pcgMaxIterations = pcgMaxIterations
        if pcgCheckEvery is not None: t.pcgCheckEvery = pcgCheckEvery
        if profilePhases is not None: t.reserved = (t.reserved & ~1) | int(bool(profilePhases))
        if dataflowSweepsOnly is not None: t.reserved = (t.reserved & ~2) | (2 if dataflowSweepsOnly else 0)
        if islandSolves is not None: t.reserved = (t.reserved & ~4) | (0 if islandSolves else 4)
        if islandTiersOff is not None: t.reserved = (t.reserved & ~0xF0) | ((int(islandTiersOff) & 0xF) << 4)
        if islandBigTier is not None: t.reserved = (t.reserved & ~256) | (256 if islandBigTier else 0)
        if svdWarmStart is not None: t.reserved = (t.reserved & ~512) | (0 if svdWarmStart else 512)
        if pbdColourBatches is not None: t.reserved = (t.reserved & ~1024) | (1024 if pbdColourBatches else 0)
        self._tuning = t
        self._ck(lib().pies_b200_set_tuning(self.h, C.byref(t)))

    def setStream(self, cuda_stream_ptr):
        self._ck(lib().pies_b200_set_stream(self.h, _vp(cuda_stream_ptr)))

    def getOptions(self):
        o = SolverOptions()
        self._ck(lib().pies_b200_get_options(self.h, C.byref(o)))
        return o

    # -- stepping (Solver.h:61-63) --
    def tick(self, deltaTime=0.0):
        self._ck(lib().pies_b200_tick(self.h, deltaTime))

    def tickPD(self, deltaTime=0.0):
        self._ck(lib().pies_b200_tick_pd(self.h, deltaTime))

    def tickPBD(self, deltaTime=0.0):
        self._ck(lib().pies_b200_tick_pbd(self.h, deltaTime))

    def tickN(self, n):
        self._ck(lib().pies_b200_tick_n(self.h, n))

    def clear(self):
        self._ck(lib().pies_b200_clear(self.h))

    releaseHinge = property(lambda self: None, lambda self, v: self._ck(lib().pies_b200_set_release_hinge(self.h, int(v))))
    renderStateDirty = property(lambda self: bool(lib().pies_b200_get_render_state_dirty(self.h)),
                                lambda self, v: self._ck(lib().pies_b200_set_render_state_dirty(self.h, int(v))))
    simFailed = property(lambda self: bool(lib().pies_b200_sim_failed(self.h)))

    # -- readback (Solver.h:65-69) --
    def getVertices(self, copy=True):
        """Solver::getVertices (Solver.h:65).  copy=False hands out a view of the solver-owned mirror, valid until
        the next mutating call - the reference's `const std::vector<Vertex>&` contract."""
        n = lib().pies_b200_vertex_count(self.h)
        if n == 0:
            return np.zeros(0, VERTEX_DTYPE)
        p = lib().pies_b200_get_vertices(self.h)
        buf = (C.c_char * (n * VERTEX_DTYPE.itemsize)).from_address(p)
        a = np.frombuffer(buf, dtype=VERTEX_DTYPE, count=n)
        return a.copy() if copy else a

    def getLines(self):
        n = lib().pies_b200_line_index_count(self.h)
        if n == 0:
            return np.zeros(0, np.uint32)
        buf = (C.c_uint32 * n).from_address(lib().pies_b200_get_lines(self.h))
        return np.frombuffer(buf, dtype=np.uint32, count=n).copy()

    def getTriangles(self):
        n = lib().pies_b200_triangle_count(self.h)
        if n == 0:
            return np.zeros((0, 3), np.uint32)
        buf = (C.c_uint32 * (3 * n)).from_address(lib().pies_b200_get_triangles(self.h))
        return np.frombuffer(buf, dtype=np.uint32, count=3 * n).reshape(n, 3).copy()

    # -- factories (Solver.h:76-116) --
    def addNodes(self, vertices):
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
        self._ck(lib().pies_b200_add_nodes(self.h, len(v), v))

    def createBox(self, translation, scale, w):
        self._ck(lib().pies_b200_create_box(self.h, _v3(translation), scale, w))

    def createTetBox(self, translation, scale, initialVelocity, w, mass, hinged=False):
        self._ck(lib().pies_b200_create_tet_box(self.h, _v3(translation), scale, _v3(initialVelocity), w, mass, int(hinged)))

    def createSheet(self, translation, scale, mass, k):
        self._ck(lib().pies_b200_create_sheet(self.h, _v3(translation), scale, mass, k))

    def createShapeMatchingBox(self, translation, countX, countY, countZ, scale, initialVelocity, w):
        self._ck(lib().pies_b200_create_shape_matching_box(self.h, _v3(translation), countX, countY, countZ, scale,
                                                          _v3(initialVelocity), w))

    def createShapeMatchingSheet(self, translation, scale, initialVelocity, w):
        self._ck(lib().pies_b200_create_shape_matching_sheet(self.h, _v3(translation), scale, _v3(initialVelocity), w))

    def createBendSheet(self, translation, scale, w):
        self._ck(lib().pies_b200_create_bend_sheet(self.h, _v3(translation), scale, w))

    def addTetMeshVolume(self, points, tets, boundaryTris, initialVelocity, density, strainStiffness, minStrain,
                         maxStrain, volumeStiffness, compression, stretching):
        """Post-TetGen half of Solver::addTriMeshVolume (PrimitiveUtilities.cpp:243-327)."""
        p = np.ascontiguousarray(points, dtype=np.float32).reshape(-1, 3)
        t = np.ascontiguousarray(tets, dtype=np.uint32).reshape(-1, 4)
        b = np.ascontiguousarray(boundaryTris, dtype=np.uint32).reshape(-1, 3)
        self._ck(lib().pies_b200_add_tet_mesh_volume(self.h, len(p), p, len(t), t.reshape(-1), len(b), b.reshape(-1),
                                                    _v3(initialVelocity), density, strainStiffness, minStrain,
                                                    maxStrain, volumeStiffness, compression, stretching))

    def addFixedRegions(self, regionMatrices, w):
        m = np.ascontiguousarray(regionMatrices, dtype=np.float32).reshape(-1, 16)
        self._ck(lib().pies_b200_add_fixed_regions(self.h, len(m), m, w))

    def updateFixedRegions(self, regionMatrices):
        m = np.ascontiguousarray(regionMatrices, dtype=np.float32).reshape(-1, 16)
        self._ck(lib().pies_b200_update_fixed_regions(self.h, len(m), m))

    def addLinkedRegions(self, regionMatrices, w):
        m = np.ascontiguousarray(regionMatrices, dtype=np.float32).reshape(-1, 16)
        self._ck(lib().pies_b200_add_linked_regions(self.h, len(m), m, w))

    # -- additive bulk builders --
    def appendNodes(self, pos, vel=None, radius=0.1, invMass=1.0):
        p = np.ascontiguousarray(pos, dtype=np.float32).reshape(-1, 3)
        n = len(p)
        v = np.zeros_like(p) if vel is None else np.ascontiguousarray(vel, dtype=np.float32).reshape(-1, 3)
        r = np.ascontiguousarray(np.broadcast_to(np.asarray(radius, np.float32), (n,)))
        m = np.ascontiguousarray(np.broadcast_to(np.asarray(invMass, np.float32), (n,)))
        first = C.c_uint32()
        self._ck(lib().pies_b200_append_nodes(self.h, n, p, v, r, m, C.byref(first)))
        return first.value

    def appendDistanceConstraints(self, ids, w):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1, 2)
        self._ck(lib().pies_b200_append_distance_constraints(self.h, len(a), a.reshape(-1), w))

    def appendPositionConstraints(self, ids, w):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1)
        self._ck(lib().pies_b200_append_position_constraints(self.h, len(a), a, w))

    def appendTetConstraints(self, ids, w, minStrain=0.8, maxStrain=1.0):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1, 4)
        self._ck(lib().pies_b200_append_tet_constraints(self.h, len(a), a.reshape(-1), w, minStrain, maxStrain))

    def appendVolumeConstraints(self, ids, w, compression=1.0, stretching=1.0):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1, 4)
        self._ck(lib().pies_b200_append_volume_constraints(self.h, len(a), a.reshape(-1), w, compression, stretching))

    def appendBendConstraints(self, ids, w):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1, 4)
        self._ck(lib().pies_b200_append_bend_constraints(self.h, len(a), a.reshape(-1), w))

    def appendShapeConstraint(self, ids, w):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1)
        self._ck(lib().pies_b200_append_shape_constraint(self.h, len(a), a, w))

    def appendTriangles(self, ids):
        a = np.ascontiguousarray(ids, dtype=np.uint32).reshape(-1, 3)
        self._ck(lib().pies_b200_append_triangles(self.h, len(a), a.reshape(-1)))

    # -- additive state access --
    def _vec(self, fn):
        out = np.empty((lib().pies_b200_vertex_count(self.h), 3), dtype=np.float32)
        self._ck(fn(self.h, out))
        return out

    positions = property(lambda self: self._vec(lib().pies_b200_get_positions))
    prevPositions = property(lambda self: self._vec(lib().pies_b200_get_prev_positions))
    velocities = property(lambda self: self._vec(lib().pies_b200_get_velocities))

    def getState(self, pos=None, prev=None, vel=None):
        """Reads the node state into caller-owned C-contiguous float32 (n, 3) arrays (pinned or pageable)."""
        n = lib().pies_b200_vertex_count(self.h)
        for a, fn in ((pos, lib().pies_b200_get_positions), (prev, lib().pies_b200_get_prev_positions),
                      (vel, lib().pies_b200_get_velocities)):
            if a is None:
                continue
            if a.dtype != np.float32 or not a.flags.c_contiguous or a.size != 3 * n:
                raise ValueError("getState needs C-contiguous float32 arrays of %d x 3" % n)
            self._ck(fn(self.h, a))

    def setState(self, pos=None, prev=None, vel=None):
        arrs = [None if a is None else np.ascontiguousarray(a, dtype=np.float32) for a in (pos, prev, vel)]
        ptrs = [None if a is None else a.ctypes.data_as(_vp) for a in arrs]
        self._ck(lib().pies_b200_set_state(self.h, *ptrs))

    def detect(self):
        self._ck(lib().pies_b200_detect(self.h))

    def triCollisions(self):
        out = np.empty((lib().pies_b200_tri_collision_count(self.h), 4), dtype=np.uint32)
        self._ck(lib().pies_b200_get_tri_collisions(self.h, out))
        return out

    def collisionCsr(self):
        """(cPtr, cCol, cVal, cDiag): the collision terms of the last detection as the CG mat-vec streams them."""
        n = lib().pies_b200_vertex_count(self.h)
        nnz = C.c_uint64(0)
        ptr = np.zeros(n + 1, np.int32); diag = np.zeros(n, np.float32)
        p = lambda a: a.ctypes.data_as(_vp)
        self._ck(lib().pies_b200_get_collision_csr(self.h, C.byref(nnz), p(ptr), None, None, p(diag)))
        col = np.zeros(nnz.value, np.int32); val = np.zeros(nnz.value, np.float32)
        if nnz.value:
            self._ck(lib().pies_b200_get_collision_csr(self.h, C.byref(nnz), None, p(col), p(val), None))
        return ptr, col, val, diag

    def debugIslandTrace(self, slot):
        """Diagnostics: (rows, iterations, SM clocks, matrix entries) per island of list `slot` in the last global solve
        (PIES_B200_ISLAND_TRACE must be set in the environment before the first tick)."""
        cnt = C.c_uint32(0)
        self._ck(lib().pies_b200_debug_island_trace(self.h, int(slot), None, 0, C.byref(cnt)))
        out = np.zeros((cnt.value, 4), np.uint32)
        if cnt.value:
            self._ck(lib().pies_b200_debug_island_trace(self.h, int(slot), out.ctypes.data_as(C.c_void_p), cnt.value, C.byref(cnt)))
        return out

    def setColliders(self, colliders):
        """Replaces the static colliders (a list of Collider, e.g. from halfspace / sphere / box; [] removes all)."""
        colliders = list(colliders)
        self._ck(lib().pies_b200_set_colliders(self.h, len(colliders), C.cast(_collider_array(colliders), _vp)))

    def colliderContacts(self):
        """Per node, the collider contact mask of the last PD detection (bit k = in contact with collider k)."""
        out = np.zeros(lib().pies_b200_vertex_count(self.h), np.uint32)
        if len(out):
            self._ck(lib().pies_b200_get_collider_contacts(self.h, out))
        return out

    def setDragTargets(self, nodes, targets, weights):
        """Replaces the drag targets: node ids, their targets (n x 3) and weights (n,).  Empty arrays remove the set."""
        ids = np.ascontiguousarray(nodes, dtype=np.uint32).reshape(-1)
        g = np.ascontiguousarray(targets, dtype=np.float32).reshape(-1, 3)
        w = np.ascontiguousarray(np.broadcast_to(np.asarray(weights, np.float32), ids.shape))
        if len(g) != len(ids):
            raise ValueError("setDragTargets: %d nodes but %d targets" % (len(ids), len(g)))
        p = lambda a: a.ctypes.data_as(_vp) if a.size else None
        self._ck(lib().pies_b200_set_drag_targets(self.h, len(ids), p(ids), p(g), p(w)))

    def raycast(self, origins, dirs, tMax=np.inf):
        """Closest hit of each ray o + t d (0 <= t <= tMax) against the triangles at the current positions:
        (tri int32 (n,), -1 on a miss; t float32 (n,), +inf on a miss; uv float32 (n, 2), the barycentric weights of
        corners 1 and 2 of the hit triangle)."""
        o = np.ascontiguousarray(origins, dtype=np.float32).reshape(-1, 3)
        d = np.ascontiguousarray(dirs, dtype=np.float32).reshape(-1, 3)
        n = len(o)
        if len(d) != n:
            raise ValueError("raycast: %d origins but %d directions" % (n, len(d)))
        tm = np.ascontiguousarray(np.broadcast_to(np.asarray(tMax, np.float32), (n,)))
        tri = np.full(n, -1, np.int32); t = np.full(n, np.inf, np.float32); uv = np.zeros((n, 2), np.float32)
        p = lambda a: a.ctypes.data_as(_vp) if a.size else None
        self._ck(lib().pies_b200_raycast(self.h, n, p(o), p(d), p(tm), p(tri), p(t), p(uv)))
        return tri, t, uv

    def setExternalForces(self, nodes, forces):
        """Replaces the host forces: node ids and their forces (n x 3), applied every substep until replaced.  Empty
        arrays remove the set."""
        ids = np.ascontiguousarray(nodes, dtype=np.uint32).reshape(-1)
        f = np.ascontiguousarray(forces, dtype=np.float32).reshape(-1, 3)
        if len(f) != len(ids):
            raise ValueError("setExternalForces: %d nodes but %d forces" % (len(ids), len(f)))
        p = lambda a: a.ctypes.data_as(_vp) if a.size else None
        self._ck(lib().pies_b200_set_external_forces(self.h, len(ids), p(ids), p(f)))

    def setWind(self, velocity, normalDrag, tangentialDrag):
        """Sets a uniform wind acting on the triangles: its velocity (3,) and the normal and tangential drag coefficients
        (both 0 removes it)."""
        w = _v3(velocity)
        self._ck(lib().pies_b200_set_wind(self.h, w.ctypes.data_as(_vp), normalDrag, tangentialDrag))

    def externalForces(self):
        """Per node, the external force (host force plus wind, gravity excluded) applied in the last substep of the
        last tick: float32 (n, 3)."""
        out = np.zeros((lib().pies_b200_vertex_count(self.h), 3), np.float32)
        if len(out):
            self._ck(lib().pies_b200_get_external_forces(self.h, out.ctypes.data_as(_vp)))
        return out

    def staticCollisions(self):
        out = np.empty(lib().pies_b200_static_collision_count(self.h), dtype=np.uint32)
        self._ck(lib().pies_b200_get_static_collisions(self.h, out))
        return out

    def triOccupancy(self):
        nc, nm = C.c_uint64(), C.c_uint64()
        self._ck(lib().pies_b200_tri_occupancy_counts(self.h, C.byref(nc), C.byref(nm)))
        cells = np.empty((nc.value, 3), np.int64); counts = np.empty(nc.value, np.uint32)
        members = np.empty(nm.value, np.uint32)
        if nc.value:
            self._ck(lib().pies_b200_get_tri_occupancy(self.h, cells, counts, members))
        return cells, counts, members

    # ---- tick phases / halo support (slab-partitioned hosts, pies_b200/multigpu.py) ----
    def pdTickBegin(self):
        self._ck(lib().pies_b200_pd_tick_begin(self.h))

    def pdSubstepBegin(self):
        self._ck(lib().pies_b200_pd_substep_begin(self.h))

    def pdIteration(self):
        self._ck(lib().pies_b200_pd_iteration(self.h))

    def pdSubstepEnd(self):
        self._ck(lib().pies_b200_pd_substep_end(self.h))

    def pdTickEnd(self):
        self._ck(lib().pies_b200_pd_tick_end(self.h))

    def deviceState(self):
        """(q_ptr, prev_ptr, vel_ptr, n): raw device addresses of the float4 node-state planes."""
        q, p, v, n = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_uint32()
        self._ck(lib().pies_b200_device_state(self.h, C.byref(q), C.byref(p), C.byref(v), C.byref(n)))
        return q.value, p.value, v.value, n.value

    def setTriangleOrder(self, order):
        if order is None:
            self._ck(lib().pies_b200_set_triangle_order(self.h, 0, np.zeros(1, np.uint32)))
        else:
            order = np.ascontiguousarray(order, np.uint32)
            self._ck(lib().pies_b200_set_triangle_order(self.h, len(order), order))

    def setOwnedNodes(self, mask):
        mask = np.ascontiguousarray(mask, np.uint8)
        self._ck(lib().pies_b200_set_owned_nodes(self.h, len(mask), mask))

    # -- render interop (include/pies_b200.h) --
    def setVertexBuffer(self, device_ptr):
        """device_ptr: a caller-owned device buffer of vertex_count x 36 bytes (e.g. an imported render buffer), or None."""
        self._ck(lib().pies_b200_set_vertex_buffer(self.h, _vp(device_ptr) if device_ptr else None))

    def deviceVertices(self):
        """(device pointer, count) of the up-to-date Vertex array on the device; no host copy."""
        p, n = C.c_void_p(), C.c_uint32()
        self._ck(lib().pies_b200_device_vertices(self.h, C.byref(p), C.byref(n)))
        return p.value, n.value

    # -- multi-GPU halo inside the library (include/pies_b200.h: pies_b200_halo_*) --
    @staticmethod
    def haloUniqueId():
        """128 bytes from ncclGetUniqueId (call on one rank, broadcast to all)."""
        buf = C.create_string_buffer(128)
        rc = lib().pies_b200_halo_unique_id(C.cast(buf, _vp))
        if rc != 0:
            raise PiesError("pies_b200_halo_unique_id failed (%d): %s" % (rc, lib().pies_b200_last_error(None).decode()))
        return buf.raw

    def haloInit(self, rank, world, unique_id):
        buf = C.create_string_buffer(bytes(unique_id), 128)
        self._ck(lib().pies_b200_halo_init(self.h, rank, world, C.cast(buf, _vp)))

    def haloSetLists(self, send, recv):
        """send / recv: dicts peer -> local row indices (pies_b200.multigpu.SlabPlan.exchange_lists)."""
        peers = sorted(set(send) | set(recv))
        e = np.zeros(0, np.uint32)
        sc = np.array([len(send.get(p, e)) for p in peers], np.uint32)
        rcnt = np.array([len(recv.get(p, e)) for p in peers], np.uint32)
        si = np.ascontiguousarray(np.concatenate([np.asarray(send.get(p, e), np.uint32) for p in peers]) if peers else e)
        ri = np.ascontiguousarray(np.concatenate([np.asarray(recv.get(p, e), np.uint32) for p in peers]) if peers else e)
        pa = np.ascontiguousarray(peers, np.int32)
        ptr = lambda a: a.ctypes.data_as(_vp) if len(a) else None
        self._ck(lib().pies_b200_halo_set_lists(self.h, len(peers), ptr(pa), ptr(sc), ptr(si), ptr(rcnt), ptr(ri)))

    def haloExchange(self, planes):
        self._ck(lib().pies_b200_halo_exchange(self.h, planes))

    def haloDestroy(self):
        self._ck(lib().pies_b200_halo_destroy(self.h))

    def countOwnedContacts(self):
        a, b = C.c_uint32(), C.c_uint32()
        self._ck(lib().pies_b200_count_owned_contacts(self.h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def detectNodes(self):
        self._ck(lib().pies_b200_detect_nodes(self.h))

    def nodeOccupancy(self):
        """Node-hash cells of the last PBD iteration: (cells[nc,3] sorted by (x,y,z), counts[nc], members ascending per cell)."""
        nc, nm = C.c_uint64(), C.c_uint64()
        self._ck(lib().pies_b200_node_occupancy_counts(self.h, C.byref(nc), C.byref(nm)))
        cells = np.empty((nc.value, 3), np.int64); counts = np.empty(nc.value, np.uint32)
        members = np.empty(nm.value, np.uint32)
        if nc.value:
            self._ck(lib().pies_b200_get_node_occupancy(self.h, cells, counts, members))
        return cells, counts, members

    def stats(self):
        st = Stats()
        self._ck(lib().pies_b200_get_stats(self.h, C.byref(st)))
        return st


# ---- probes (module-level: they need no solver) ----
def _ckp(rc):
    if rc != 0:
        raise PiesError("pies_b200 probe failed: %d" % rc)


def probe_tet_projection(pos, qinv, minStrain, maxStrain):
    pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 12); qinv = np.ascontiguousarray(qinv, np.float32).reshape(-1, 9)
    out = np.empty_like(pos)
    _ckp(lib().pies_b200_probe_tet_projection(len(pos), pos, qinv, minStrain, maxStrain, out))
    return out


def probe_volume_projection(pos, qinv, minOmega, maxOmega):
    pos = np.ascontiguousarray(pos, np.float32).reshape(-1, 12); qinv = np.ascontiguousarray(qinv, np.float32).reshape(-1, 9)
    out = np.empty_like(pos)
    _ckp(lib().pies_b200_probe_volume_projection(len(pos), pos, qinv, minOmega, maxOmega, out))
    return out


def probe_ccd(queries, threshold):
    q = np.ascontiguousarray(queries, np.float32).reshape(-1, 18)
    hit = np.empty(len(q), np.int32); t = np.empty(len(q), np.float32)
    _ckp(lib().pies_b200_probe_ccd(len(q), q, threshold, hit, t))
    return hit, t


def probe_edge_ccd(queries):
    q = np.ascontiguousarray(queries, np.float32).reshape(-1, 18)
    hit = np.empty(len(q), np.int32); t = np.empty(len(q), np.float32)
    _ckp(lib().pies_b200_probe_edge_ccd(len(q), q, hit, t))
    return hit, t


def probe_tri_range(pos, prev):
    p = np.ascontiguousarray(pos, np.float32).reshape(-1, 9); o = np.ascontiguousarray(prev, np.float32).reshape(-1, 9)
    mins = np.empty((len(p), 3), np.int64); lens = np.empty((len(p), 3), np.uint32)
    _ckp(lib().pies_b200_probe_tri_range(len(p), p, o, mins, lens))
    return mins, lens


def probe_node_range(pos, radius, gridScale):
    p = np.ascontiguousarray(pos, np.float32).reshape(-1, 3); r = np.ascontiguousarray(radius, np.float32).reshape(-1)
    mins = np.empty((len(p), 3), np.int64); lens = np.empty((len(p), 3), np.uint32)
    _ckp(lib().pies_b200_probe_node_range(len(p), p, r, gridScale, mins, lens))
    return mins, lens


def probe_sort_pairs(keys, vals, keyBits):
    k = np.ascontiguousarray(keys, np.uint64).copy(); v = np.ascontiguousarray(vals, np.uint32).copy()
    _ckp(lib().pies_b200_probe_sort_pairs(len(k), k, v, keyBits))
    return k, v


def probe_sell(rowPtr, col, val):
    """Host-only: the sliced-ELLPACK copy (sellPtr, sellRow, sellCol, sellVal) the CG mat-vec reads, from a CSR matrix."""
    rp = np.ascontiguousarray(rowPtr, np.int32); c = np.ascontiguousarray(col, np.int32); v = np.ascontiguousarray(val, np.float32)
    n = len(rp) - 1
    padded = C.c_uint64(0)
    p = lambda a: a.ctypes.data_as(_vp)
    _ckp(lib().pies_b200_probe_sell(n, p(rp), p(c), p(v), None, None, None, None, C.byref(padded)))
    ns = (n + 31) // 32
    sp = np.zeros(ns + 1, np.uint32); sr = np.zeros(32 * ns, np.uint32)
    sc = np.zeros(padded.value, np.int32); sv = np.zeros(padded.value, np.float32)
    _ckp(lib().pies_b200_probe_sell(n, p(rp), p(c), p(v), p(sp), p(sr), p(sc), p(sv), C.byref(padded)))
    return sp, sr, sc, sv


def probe_colliders(points, colliders):
    """(phi[nPoints, nColliders], normals[nPoints, nColliders, 3]) of the library's device functions."""
    p = np.ascontiguousarray(points, np.float32).reshape(-1, 3)
    colliders = list(colliders)
    phi = np.zeros((len(p), len(colliders)), np.float32)
    nrm = np.zeros((len(p), len(colliders), 3), np.float32)
    rc = lib().pies_b200_probe_colliders(len(p), p.ctypes.data_as(_vp), len(colliders), C.cast(_collider_array(colliders), _vp),
                                         phi.ctypes.data_as(_vp), nrm.ctypes.data_as(_vp))
    if rc != 0:
        raise PiesError("pies_b200_probe_colliders failed: %d" % rc)
    return phi, nrm


def probe_segments(cmds, mesh_points=None, mesh_tets=None):
    """Host-only: the closed segments of the fused local step + RHS for a scene built from commands (rows of
    kind, tx, ty, tz, a, b, c, d; see pies_b200_probe_segments), with the gather lists they were cut from."""
    cm = np.ascontiguousarray(cmds, np.float32).reshape(-1, 8)
    mp = None if mesh_points is None else np.ascontiguousarray(mesh_points, np.float32).reshape(-1, 3)
    mt = None if mesh_tets is None else np.ascontiguousarray(mesh_tets, np.uint32).reshape(-1, 4)
    p = lambda a: None if a is None else a.ctypes.data_as(_vp)
    head = (len(cm), p(cm), 0 if mp is None else len(mp), p(mp), 0 if mt is None else len(mt), p(mt))
    sizes = np.zeros(7, np.uint64)
    _ckp(lib().pies_b200_probe_segments(*head, sizes, *([None] * 7)))
    n, ninc, ne, ns, nre, nrn, base = (int(x) for x in sizes)
    out = dict(incPtr=np.zeros(n + 1, np.int32), inc=np.zeros(ninc, np.uint32), segSlot=np.zeros(ninc, np.uint16),
               elemIds=np.zeros((ne, 4), np.uint32), segs=np.zeros((ns, 4), np.uint32),
               restElems=np.zeros(nre, np.uint32), restNodes=np.zeros(nrn, np.uint32))
    keys = ("incPtr", "inc", "segSlot", "elemIds", "segs", "restElems", "restNodes")
    _ckp(lib().pies_b200_probe_segments(*head, sizes, *(p(out[k]) for k in keys)))
    out["baseTet"] = base
    return out
