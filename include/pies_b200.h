/* pies_b200.h — C ABI of the B200-native Pies solver loop.
 *
 * Drop-in boundary: every entry point below replaces one member of the
 * reference's only public class, Pies::Solver (reference Include/Pies/Solver.h:40-199),
 * or is an additive extension the reference has no public API for (marked
 * [additive], SURVEY F14).  The header-only C++ class in Include/Pies/Solver.h of
 * this repo forwards the reference's glm-typed signatures to these functions, so
 * a host application that used the reference recompiles unchanged and links
 * libpies_b200.so.  No torch / STL / glm types cross this boundary: plain
 * pointers, sizes and PODs only.  All functions return 0 on success and a
 * negative PIES_B200_E* code on failure; pies_b200_last_error() gives the text.
 * Nothing here falls back to the CPU: without a CUDA device create() fails.
 *
 * Threading: one caller thread per solver (same as the reference); tick() is
 * synchronous — it returns after the device has finished the tick.
 */
#ifndef PIES_B200_H
#define PIES_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PIES_B200_OK 0
#define PIES_B200_EINVAL -1   /* bad argument */
#define PIES_B200_ECUDA -2    /* CUDA runtime / launch failure (also latches simFailed) */
#define PIES_B200_ENODEV -3   /* no usable sm_100 device: there is no CPU fallback */
#define PIES_B200_ERANGE -4   /* a scene exceeds a documented limit */
#define PIES_B200_ENOCONV -5  /* the global solve stopped at pcgMaxIterations far from its tolerance (the tick completed; see stats) */

/* Mirrors Pies::SolverOptions field for field, same defaults
 * (reference Include/Pies/Solver.h:23-38); solver: 0 = PBD, 1 = PD
 * (SolverName, Solver.h:21). */
typedef struct PiesB200Options {
  float fixedTimestepSize;                   /* 0.012 */
  uint32_t timeSubsteps;                     /* 1 */
  uint32_t iterations;                       /* 4 */
  uint32_t collisionStabilizationIterations; /* 4 */
  float collisionThresholdDistance;          /* 0.1 */
  float collisionThickness;                  /* 0.05 */
  float gravity;                             /* 10 */
  float damping;                             /* 0.006 */
  float friction;                            /* 0.01 */
  float staticFrictionThreshold;             /* 0 */
  float floorHeight;                         /* 0 */
  float gridSpacing;                         /* 2 */
  uint32_t threadCount;                      /* 8: fixes the canonical order of the collision lists (SURVEY F8) */
  uint32_t solver;                           /* 1 = PD */
} PiesB200Options;

/* Mirrors Pies::Solver::Vertex (reference Include/Pies/Solver.h:42-49), 36 bytes. */
typedef struct PiesB200Vertex {
  float position[3];
  float radius;
  float baseColor[3];
  float roughness;
  float metallic;
} PiesB200Vertex;

/* Solver knobs the reference does not have (its global step is a direct sparse
 * Cholesky, Solver.cpp:213-215,258-262,356; ours is a preconditioned CG). */
typedef struct PiesB200Tuning {
  float pcgTolerance;        /* stop when ||r||_2 <= tol * ||b||_2 per coordinate column; default 1e-7 */
  uint32_t pcgMaxIterations; /* default 200 */
  uint32_t pcgCheckEvery;    /* host polls the device convergence flag every k iterations; default 1 */
  uint32_t reserved;         /* flag bits: 1 = record per-phase CUDA-event timings into PiesB200Stats (no extra syncs);
                              * 2 = ordered contact sweeps of every cluster above 32 nodes by the dataflow executor
                              *     (no shared-memory sweeps of mid-size clusters; same result, for testing);
                              * 4 = no island-local solves: every island goes to the grid-wide CG (for testing);
                              * 16 << t = island tier t (0..3) disabled: its islands move to the next tier that fits;
                              * 256 = island tier 3 enabled (one 1024-thread CTA per island of up to 7 168 nodes; off by default:
                              *       such islands go to the grid-wide CG);
                              * 1024 = PBD node-node response in colour batches instead of the reference's sequential order
                              *       (same operation per pair and per visit, different visiting order: for scenes whose contact
                              *       graph is one long chain, where the exact order is inherently serial; see pbd.cu);
                              * 512 = cold-start the 3x3 SVD of every tet projection (no warm start from the previous iteration's
                              *       factors: same result up to rounding, for testing) */
} PiesB200Tuning;

/* Counters and device-side phase timings of the most recent tick ([additive]). */
typedef struct PiesB200Stats {
  uint64_t staticProjections;    /* static constraint projections per PD iteration (shape/goal count one per member) */
  uint64_t collisionProjections; /* live point-triangle + floor constraints of the last substep */
  uint64_t projectionsLastTick;  /* sum over substeps and iterations of (static + live collision) */
  uint64_t pcgIterationsLastTick;
  uint64_t kernelLaunchesLastTick;
  uint32_t triCollisions;
  uint32_t staticCollisions;
  uint32_t substepsLastTick;
  uint32_t simFailed;
  float msTick;        /* CUDA-event time of the whole tick on the solver stream */
  float msLocal;       /* local projections + RHS gather (sum over iterations) */
  float msGlobal;      /* PCG global solve */
  float msDetect;      /* spatial hash + CCD */
  float msContact;     /* stabilisation + friction */
  float msOther;
  float pcgLastRelResidual;
  float msTetKernel;           /* time inside the fused tet strain+volume projection kernel alone */
  uint32_t tetKernelLaunches;  /* its launches in the last tick */
  uint32_t reserved;           /* contact clusters of the last substep swept from shared memory (low 16 bits, saturating)
                                * and by the dataflow executor (high 16 bits) */
  /* sampled launches of the other hot kernels (one timed launch per PD iteration; phase timing on only) */
  float msSpmvKernel;          /* k_pcg_spmv: A z (SELL windows) + p / Ap recurrences */
  float msUpdateKernel;        /* k_pcg_update: x, r update + block-Jacobi apply */
  float msGatherKernel;        /* k_gather_rhs: CSR gather of the right-hand side */
  uint32_t spmvKernelLaunches;
  uint32_t updateKernelLaunches;
  uint32_t gatherKernelLaunches;
  /* global solve by islands (connected components of S + C_t), last substep: islands solved by one warp / one CTA
   * (tiers 0..3) and islands, with their node count, left to the grid-wide CG */
  uint32_t islandsTier[4];
  uint32_t islandsGlobal;
  uint32_t islandNodesGlobal;
  /* solves of the last tick (island-local or grid-wide) that stopped at pcgMaxIterations instead of the tolerance,
   * and the worst relative residual among them (0 when none) */
  uint32_t pcgCapHits;
  float pcgWorstCapResidual;
  float msIslandKernels;       /* time inside the island-local solve kernels (phase timing on only) */
  uint32_t islandKernelLaunches;
  uint64_t pcgIslandRowIterations; /* sum over island solves of iterations x ceil(rows / 32): the work the island kernels did */
  /* slab-partitioned runs (pies_b200_halo_*): bytes sent + received, exchanges and device time of the halo exchanges */
  uint64_t haloBytesLastTick;
  uint32_t haloExchangesLastTick;
  float msHalo;
  uint64_t systemNonZeros;     /* non-zeros of S = M/h^2 + sum w A^T A (both triangles), for the CG byte model */
  uint32_t staticBodies;       /* connected components of S */
  uint32_t islandInverseFloats; /* floats of block / dense inverse one global solve of the island lists reads (last substep) */
} PiesB200Stats;

typedef struct PiesB200Solver PiesB200Solver;

/* ---- lifetime (Solver::Solver(const SolverOptions&), ~Solver; Solver.cpp:11-23) ---- */
void pies_b200_default_options(PiesB200Options* out);
void pies_b200_default_tuning(PiesB200Tuning* out);
/* options == NULL behaves like the reference's Solver(SolverOptions{}) (deliberate fix of the
 * default-ctor hazard, SURVEY §8b).  device < 0 selects the current CUDA device. */
int pies_b200_create(const PiesB200Options* options, int device, PiesB200Solver** out);
void pies_b200_destroy(PiesB200Solver* s);
const char* pies_b200_last_error(const PiesB200Solver* s); /* s may be NULL: last create() error */
int pies_b200_set_tuning(PiesB200Solver* s, const PiesB200Tuning* t);
/* Run on a caller-owned CUDA stream (cudaStream_t as void*), e.g. torch's current stream. */
int pies_b200_set_stream(PiesB200Solver* s, void* cudaStream);
int pies_b200_get_options(const PiesB200Solver* s, PiesB200Options* out); /* Solver::getOptions, Solver.h:71 */

/* ---- stepping (Solver::tick / tickPD / tickPBD; Solver.cpp:25-486; dt is ignored like the reference) ---- */
int pies_b200_tick(PiesB200Solver* s, float deltaTime);
int pies_b200_tick_pd(PiesB200Solver* s, float deltaTime);
int pies_b200_tick_pbd(PiesB200Solver* s, float deltaTime);
/* n ticks back to back [additive]. */
int pies_b200_tick_n(PiesB200Solver* s, uint32_t n);
int pies_b200_set_release_hinge(PiesB200Solver* s, int release); /* public member releaseHinge, Solver.h:52 */
int pies_b200_get_render_state_dirty(const PiesB200Solver* s);   /* public member renderStateDirty, Solver.h:51 */
int pies_b200_set_render_state_dirty(PiesB200Solver* s, int dirty);
int pies_b200_sim_failed(const PiesB200Solver* s);               /* the _simFailed latch, Solver.cpp:26-28,852-856 */
int pies_b200_clear(PiesB200Solver* s);                          /* Solver::clear, Solver.cpp:488-507 */

/* ---- [additive] static colliders: half-spaces, spheres and oriented solid boxes (DESIGN.md section 9).
 *      The reference has no collision geometry but the floor; a host that wants a container, a ramp or an obstacle sets
 *      them here.  Each collider k has a signed distance phi_k(x) (negative inside) and an outward normal n_k(x):
 *        half-space: phi = n . (x - c), n normalised by the library;
 *        sphere:     phi = |x - c| - r, n = (x - c) / |x - c| (n = +y at x = c);
 *        box:        the box signed distance in its local frame; outside, n points from the closest surface point to x;
 *                    inside, n is the normal of the nearest face (tie: lowest axis first, then the + side).
 *      Colliders are static during a tick and evaluated in ascending index order everywhere.  The set may be replaced
 *      between ticks (moving an obstacle rebuilds nothing).
 *      PD: a node with phi_k(q) < collisionThickness at detection is in contact with k for the substep; every iteration
 *      it is pulled towards q - min(phi_k(q), 0) n_k(q) with weight 1e4 (the floor's weight); after stabilisation it is
 *      projected out of its colliders, and friction acts along each collider's tangent plane.  The node radius is ignored,
 *      as for the PD floor.  PBD: a node with phi_k(x) < radius is pushed to phi_k = radius every iteration, and the
 *      floor's friction rule acts on the tangential velocity.
 *      Collider contacts are not counted in PiesB200Stats (the projection counters keep the reference's definition),
 *      and nothing about them is read back during a tick. ---- */
#define PIES_B200_COLLIDER_HALFSPACE 0
#define PIES_B200_COLLIDER_SPHERE 1
#define PIES_B200_COLLIDER_BOX 2
#define PIES_B200_MAX_COLLIDERS 32 /* the width of the per-node contact mask */
typedef struct PiesB200Collider { /* 64 bytes */
  uint32_t kind;                  /* PIES_B200_COLLIDER_* */
  float center[3];                /* half-space: a point on its plane; sphere, box: the centre */
  float axes[9];                  /* half-space: axes[0..2] = outward normal; box: three orthonormal axes, column after column */
  float extent[3];                /* sphere: radius in extent[0]; box: half extents */
} PiesB200Collider;
/* Replaces the solver's colliders (n = 0 removes all) between ticks.  EINVAL: unknown kind, non-finite value, zero normal,
 * radius or half extent <= 0, box axes not orthonormal within 1e-4, or a call inside pd_tick_begin .. pd_tick_end;
 * ERANGE: n > PIES_B200_MAX_COLLIDERS.  A rejected set leaves the previous one in place.  pies_b200_clear removes them. */
int pies_b200_set_colliders(PiesB200Solver* s, uint32_t n, const PiesB200Collider* c);
/* vertex_count() masks of the last PD detection (tick or pies_b200_detect): bit k = node in contact with collider k.
 * All zero when the solver had no colliders then. */
int pies_b200_get_collider_contacts(PiesB200Solver* s, uint32_t* masks);
/* The device functions of phi and n on caller data (validated like set_colliders): for point p and collider k,
 * phi[p * nColliders + k] and normals[3 * (p * nColliders + k) + 0..2]. */
int pies_b200_probe_colliders(uint32_t nPoints, const float* xyz, uint32_t nColliders, const PiesB200Collider* c,
                              float* phi, float* normals);

/* ---- [additive] picking and dragging (DESIGN.md section 10): what an interactive host needs to click a body and pull it.
 *
 * Drag targets: one-node position constraints whose target and weight the host replaces between ticks, without a
 * topology rebuild (DESIGN.md section 10).  Each call replaces the whole set (n = 0 removes it); the set persists across
 * ticks until replaced, stays valid when bodies are appended, and pies_b200_clear removes it.  The arrays are copied
 * before the call returns.  EINVAL: a node id >= vertex_count(), a duplicate id, a non-finite target or weight, a
 * weight <= 0, a null array with n > 0, or a call inside pd_tick_begin .. pd_tick_end; a rejected set leaves the
 * previous one in place.
 *   PD: each drag is a PositionConstraint of weight w and target g for the substep: w joins the node's one-node weight
 *       (after the floor's and the colliders') in the diagonal of the global step, and w g its right-hand side.
 *   PBD: every iteration, right after the position-constraint sweep (also with release_hinge), x += min(w, 1) (g - x).
 *   Drags take no part in stabilisation or friction, ignore release_hinge and are not counted in PiesB200Stats.
 *   Without a set, every kernel computes what it computed before drags existed. */
int pies_b200_set_drag_targets(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* targets /* 3n */,
                               const float* weights /* n */);
/* Closest hit of each ray o + t d, 0 <= t <= tMax[r], against the solver's triangles at the positions get_vertices()
 * returns (two-sided; d need not be normalised, t is in units of d).  tri[r] = index into get_triangles() / 3 of the hit
 * with the smallest t, ties to the lowest index, -1 on a miss; t[r] = +inf on a miss; uv[2r], uv[2r+1] = barycentric
 * weights of corners 1 and 2 of that triangle (0 on a miss).  Moller-Trumbore in fp32 (operation order in DESIGN.md
 * section 10); a triangle parallel to the ray or of zero area never hits.  Sees set_state without a tick, marks nothing
 * dirty, and returns when the results are on the host.  Cost: nRays x triangle_count() ray-triangle tests (no
 * acceleration structure).  EINVAL: a non-finite origin, a zero or non-finite direction, a NaN or negative tMax (+inf is
 * allowed), or a null array with nRays > 0.  A scene without triangles returns all misses. */
int pies_b200_raycast(PiesB200Solver* s, uint32_t nRays, const float* origins /* 3 per ray */, const float* dirs /* 3 per ray */,
                      const float* tMax, int32_t* tri, float* t, float* uv /* 2 per ray */);

/* ---- [additive] external forces (DESIGN.md section 11): per-node forces a host applies, and a uniform wind acting on the
 *      triangles.  Gravity stays as it is; the external force f_i of node i joins it where it acts:
 *        PD:  the velocity update, v_i = [the reference's expression] + (h f_i) invMass_i, so f moves the next
 *             substep's prediction, like gravity;
 *        PBD: the advection, x_i = [the reference's expression] + ((f_i invMass_i) dt) dt.
 *      (h = dt = fixedTimestepSize / timeSubsteps; each added operation rounded on its own.)  A node with invMass = 0
 *      gains nothing.  f_i is evaluated once per substep, on the positions x and velocities v at the substep start:
 *        f_i = hostForce_i + sum over the triangles t containing i, in ascending index order, of f_t / 3.
 *      Wind velocity w, normal and tangential drag coefficients c_n, c_t >= 0; for triangle t = (a, b, c), every
 *      operation rounded on its own (order in DESIGN.md section 11):
 *        m = cross(x_b - x_a, x_c - x_a); |m| = 0 -> f_t = 0;  A = |m| / 2,  n = m / |m|
 *        u = (v_a + v_b + v_c) / 3 - w;  un = dot(u, n),  ut = u - un n
 *        f_t = -A (c_n un |un| n + c_t ut)     (the same for either winding)
 *      Only triangles feel the wind: ropes, bare nodes and bodies without triangles do not.  The integration is explicit
 *      and not clamped: keep h c_n A_i |un| invMass_i well below 1 (A_i = the area of node i's triangles / 3), and
 *      likewise h c_t A_i invMass_i, or the drag overshoots and the body gains energy.
 *      Neither forces nor wind are counted in PiesB200Stats.  Without either, every kernel computes what it computed
 *      before external forces existed. */
/* Replaces the host forces (3 floats per node, n = 0 removes them).  The set persists across ticks until replaced, stays
 * valid when bodies are appended (new nodes get none), and pies_b200_clear removes it.  The arrays are copied before the
 * call returns.  EINVAL: a node id >= vertex_count(), a duplicate id, a non-finite component, a null array with n > 0, or
 * a call inside pd_tick_begin .. pd_tick_end; a rejected set leaves the previous one in place. */
int pies_b200_set_external_forces(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* forces /* 3n */);
/* Sets the wind: velocity (3 floats), c_n = normalDrag, c_t = tangentialDrag.  Both coefficients 0 remove it, and so does
 * pies_b200_clear.  EINVAL: a null velocity, a non-finite value, a negative coefficient, or a call inside
 * pd_tick_begin .. pd_tick_end; a rejected call leaves the previous wind in place. */
int pies_b200_set_wind(PiesB200Solver* s, const float* velocity /* 3 */, float normalDrag, float tangentialDrag);
/* f_i of every node (3 floats per node, vertex_count() nodes) as applied in the last substep of the last tick, gravity
 * not included.  All zeros when that tick had neither forces nor wind, before the first tick and after clear; nodes
 * appended since that tick read 0. */
int pies_b200_get_external_forces(PiesB200Solver* s, float* xyz);

/* ---- readback (Solver::getVertices/getLines/getTriangles; Solver.h:65-69) ---- */
uint32_t pies_b200_vertex_count(const PiesB200Solver* s);
uint32_t pies_b200_line_index_count(const PiesB200Solver* s);
uint32_t pies_b200_triangle_count(const PiesB200Solver* s);
/* Pointers stay valid until the next mutating call, like the reference's const refs.  The position
 * mirror is brought up to date (one D2H copy) by the first get_vertices() after a tick. */
const PiesB200Vertex* pies_b200_get_vertices(const PiesB200Solver* s);
const uint32_t* pies_b200_get_lines(const PiesB200Solver* s);
const uint32_t* pies_b200_get_triangles(const PiesB200Solver* s); /* 3 per triangle */

/* [additive] Zero-copy render interop (SURVEY section 8f-3; the reference's hosts are renderers that upload getVertices()
 * to a vertex buffer every frame, Solver.h:42-49,65).  The Vertex mirror also exists on the device, 36 B per vertex:
 * device_vertices brings its positions up to date on the solver's stream (one kernel, no host copy) and returns the
 * device pointer.  With set_vertex_buffer the host supplies that buffer itself — e.g. a Vulkan / OpenGL vertex buffer
 * imported into CUDA (cudaImportExternalMemory, cudaGraphicsMapResources): the solver then writes the vertices straight
 * into the renderer's memory.  The buffer must hold vertex_count() x 36 bytes and stay valid until replaced (NULL
 * returns to the internal one); after a topology change the static attributes are rewritten on the next call. */
int pies_b200_set_vertex_buffer(PiesB200Solver* s, void* deviceBuffer);
int pies_b200_device_vertices(PiesB200Solver* s, void** deviceVertices, uint32_t* count);

/* ---- scene construction: the reference's factories (Src/PrimitiveUtilities.cpp) ---- */
int pies_b200_add_nodes(PiesB200Solver* s, uint32_t n, const float* xyz);                      /* :42-75 */
int pies_b200_create_box(PiesB200Solver* s, const float t[3], float scale, float w);           /* :620-847 */
int pies_b200_create_tet_box(PiesB200Solver* s, const float t[3], float scale, const float v0[3],
                             float w, float mass, int hinged);                                   /* :330-618 */
int pies_b200_create_sheet(PiesB200Solver* s, const float t[3], float scale, float mass, float k); /* :849-976 */
int pies_b200_create_shape_matching_box(PiesB200Solver* s, const float t[3], uint32_t countX,
                                        uint32_t countY, uint32_t countZ, float scale,
                                        const float v0[3], float w);                             /* :985-1048 */
int pies_b200_create_shape_matching_sheet(PiesB200Solver* s, const float t[3], float scale,
                                          const float v0[3], float w);                           /* :1050-1125 */
int pies_b200_create_bend_sheet(PiesB200Solver* s, const float t[3], float scale, float w);    /* :1127-1289 */
/* The post-TetGen half of Solver::addTriMeshVolume (:243-327): the caller runs TetGen (a host-side,
 * setup-time dependency the reference vendors; the C++ wrapper does it when <tetgen.h> is available)
 * and passes its output: points, tetrahedra (4 indices each) and the boundary faces already
 * filtered and re-wound as at :249-267 (3 indices each, local to this mesh). */
int pies_b200_add_tet_mesh_volume(PiesB200Solver* s, uint32_t nPoints, const float* xyz,
                                  uint32_t nTets, const uint32_t* tetIdx, uint32_t nTris,
                                  const uint32_t* triIdx, const float v0[3], float density,
                                  float strainStiffness, float minStrain, float maxStrain,
                                  float volumeStiffness, float compression, float stretching);
/* 4x4 matrices are 16 floats, column-major (glm::mat4 memory layout). */
int pies_b200_add_fixed_regions(PiesB200Solver* s, uint32_t n, const float* mats, float w);    /* :77-112 */
int pies_b200_update_fixed_regions(PiesB200Solver* s, uint32_t n, const float* mats);          /* :114-128 */
int pies_b200_add_linked_regions(PiesB200Solver* s, uint32_t n, const float* mats, float w);   /* :130-162 */

/* ---- [additive] bulk builders: what a white-box host does with createXConstraint
 *      (reference Include/Pies/Constraints.h:155-230); rest data is taken from the
 *      current node positions exactly like those factories do. ---- */
int pies_b200_append_nodes(PiesB200Solver* s, uint32_t n, const float* pos, const float* vel,
                           const float* radius, const float* invMass, uint32_t* firstId);
int pies_b200_append_distance_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids2, float w);
int pies_b200_append_position_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w);
int pies_b200_append_tet_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids4, float w,
                                     float minStrain, float maxStrain);
int pies_b200_append_volume_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids4, float w,
                                        float compression, float stretching);
int pies_b200_append_bend_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids4, float w);
int pies_b200_append_shape_constraint(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w);
int pies_b200_append_triangles(PiesB200Solver* s, uint32_t n, const uint32_t* ids3);

/* ---- [additive] state access for parity tests and hosts that need more than getVertices ---- */
int pies_b200_get_positions(PiesB200Solver* s, float* xyz);
int pies_b200_get_prev_positions(PiesB200Solver* s, float* xyz);
int pies_b200_get_velocities(PiesB200Solver* s, float* xyz);
/* Any of pos/prev/vel may be NULL (left untouched). */
int pies_b200_set_state(PiesB200Solver* s, const float* pos, const float* prev, const float* vel);
/* Runs only the once-per-substep detection pass (reference Solver.cpp:240, :680-875) on the current state. */
int pies_b200_detect(PiesB200Solver* s);
uint32_t pies_b200_tri_collision_count(const PiesB200Solver* s);
uint32_t pies_b200_static_collision_count(const PiesB200Solver* s);
int pies_b200_get_tri_collisions(PiesB200Solver* s, uint32_t* ids4);   /* canonical reference order */
/* [additive, parity] The collision terms C_t that the last detection added to the system (what the reference adds to
 * S in Solver.cpp:242-262), in the form the CG mat-vec streams: off-diagonals as a per-node CSR, diagonal separately.
 * Call with cCol == NULL to read *nnz (and fill cPtr, n + 1 entries, and cDiag, n entries, when given). */
int pies_b200_get_collision_csr(PiesB200Solver* s, uint64_t* nnz, int32_t* cPtr, int32_t* cCol, float* cVal, float* cDiag);
int pies_b200_get_static_collisions(PiesB200Solver* s, uint32_t* ids); /* canonical reference order */
/* Triangle-hash occupancy of the last detect(): cells sorted by (x,y,z), members ascending. */
int pies_b200_tri_occupancy_counts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers);
int pies_b200_get_tri_occupancy(PiesB200Solver* s, int64_t* cellsXYZ, uint32_t* counts, uint32_t* members);
/* Node-hash occupancy (SpatialHash<Node>, reference Solver.cpp:81-82) of the last PBD iteration, same layout. */
int pies_b200_detect_nodes(PiesB200Solver* s); /* rebuilds only the node hash on the current state */
int pies_b200_node_occupancy_counts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers);
int pies_b200_get_node_occupancy(PiesB200Solver* s, int64_t* cellsXYZ, uint32_t* counts, uint32_t* members);
int pies_b200_get_stats(const PiesB200Solver* s, PiesB200Stats* out);

/* ---- [additive] slab-partitioned (multi-GPU) hosts: one solver per GPU holds the bodies of its slab plus ghost
 *      copies of the neighbouring slabs' boundary bodies; between the phases below the host overwrites the ghost
 *      nodes in the device state arrays with their owners' values (NCCL).  pies_b200_tick_pd() is exactly
 *      begin; per substep { substep_begin; iterations x iteration; substep_end }; end.
 *      (reference Solver::tickPD, Solver.cpp:162-486: :229-262 / :264-365 / :367-484) ---- */
int pies_b200_pd_tick_begin(PiesB200Solver* s);
int pies_b200_pd_substep_begin(PiesB200Solver* s); /* inertia, detection, preconditioner blocks */
int pies_b200_pd_iteration(PiesB200Solver* s);     /* one local/global iteration */
int pies_b200_pd_substep_end(PiesB200Solver* s);   /* stabilisation, velocity update, friction */
int pies_b200_pd_tick_end(PiesB200Solver* s);
/* Device pointers of the node state: float4 per node, q = (x,y,z,invMass), prev = (x,y,z,radius), vel = (vx,vy,vz,0). */
int pies_b200_device_state(PiesB200Solver* s, void** q, void** prev, void** vel, uint32_t* n);
/* order[t] = position of local triangle t in the canonical collision-list order (SURVEY F8) of the GLOBAL scene
 * restricted to the local triangles; NULL restores the local thread striping. */
int pies_b200_set_triangle_order(PiesB200Solver* s, uint32_t n, const uint32_t* order);
/* mask[i] != 0: node i is owned by this solver (others are ghosts); only used for counting. */
int pies_b200_set_owned_nodes(PiesB200Solver* s, uint32_t n, const uint8_t* mask);
int pies_b200_count_owned_contacts(PiesB200Solver* s, uint32_t* nTri, uint32_t* nFloor);

/* ---- [additive] multi-GPU inside the library: NCCL halo exchange of a slab-partitioned scene (SURVEY section 8e; the
 *      reference is single-process, so this replaces nothing in it).  One process (or thread) per GPU; each solver holds
 *      its slab's bodies plus ghost copies of the neighbours' boundary bodies, created in global body order.  After
 *      halo_init + halo_set_lists, pies_b200_tick() itself overwrites the ghost rows with their owners' values at every
 *      substep start (position, previous position, velocity) and after every local/global iteration (position), and all
 *      ranks stop together if one fails.  NCCL is dlopen-ed (libnccl.so.2); without it halo_init fails. ---- */
int pies_b200_halo_unique_id(void* out128);                       /* ncclGetUniqueId: call on one rank, hand the 128 bytes to all */
int pies_b200_halo_init(PiesB200Solver* s, int rank, int world, const void* id128);  /* collective: ncclCommInitRank */
/* peers[k]: rank of the k-th slab neighbour; sendIdx holds, peer after peer, the local rows that are ghosts on that peer
 * (sendCounts[k] of them), recvIdx the local ghost rows owned by it; both sides list shared bodies in global order. */
int pies_b200_halo_set_lists(PiesB200Solver* s, int nPeers, const int* peers, const uint32_t* sendCounts,
                             const uint32_t* sendIdx, const uint32_t* recvCounts, const uint32_t* recvIdx);
int pies_b200_halo_exchange(PiesB200Solver* s, int planes);      /* explicit exchange, planes = 1 or 3 (tick() does this itself) */
int pies_b200_halo_destroy(PiesB200Solver* s);

/* Diagnostics (needs PIES_B200_ISLAND_TRACE in the environment before the first tick): the island-local solve's record
 * of the LAST global solve for list `slot` (0 warp, 1 CTA-320, 2 CTA-512, 3 CTA-1024, 4 CTA-128, 5 dense <= 128 nodes, 6 dense <= 192 nodes): four words per island —
 * rows, CG iterations, SM clocks, matrix entries.  *count receives the number of islands in the list. */
int pies_b200_debug_island_trace(PiesB200Solver* s, int slot, uint32_t* out4, uint32_t cap, uint32_t* count);

/* ---- [additive] per-kernel probes: run the device functions of the hot kernels on caller data ---- */
/* Tet strain / volume projections (reference Constraints.cpp:76-128, :205-255): pos 12 floats,
 * qinv 9 floats column-major per tet; out 12 floats (projected[0..3]). */
int pies_b200_probe_tet_projection(uint32_t n, const float* pos, const float* qinv, float minStrain,
                                   float maxStrain, float* out);
int pies_b200_probe_volume_projection(uint32_t n, const float* pos, const float* qinv, float minOmega,
                                      float maxOmega, float* out);
/* pointTriangleCCD (reference CollisionDetection.cpp:227-302): in 18 floats per query. */
int pies_b200_probe_ccd(uint32_t n, const float* in18, float threshold, int32_t* hit, float* t);
/* edgeEdgeCCD (reference CollisionDetection.cpp:304-418; never emitted by the reference's tick, SURVEY F13):
 * in 18 floats per query (ab0 ac0 ad0 ab1 ac1 ad1). */
int pies_b200_probe_edge_ccd(uint32_t n, const float* in18, int32_t* hit, float* t);
/* TriCompRange / NodeCompRange (reference Solver.cpp:942-979, :877-901). */
int pies_b200_probe_tri_range(uint32_t n, const float* pos9, const float* prev9, int64_t* mins, uint32_t* lens);
int pies_b200_probe_node_range(uint32_t n, const float* pos3, const float* radius, float gridScale,
                               int64_t* mins, uint32_t* lens);
/* Stable LSD radix sort used by the cell tables (64-bit keys, 32-bit payload). */
int pies_b200_probe_sort_pairs(uint64_t n, uint64_t* keys, uint32_t* vals, int keyBits);
/* Host-only (no device needed): the sliced-ELLPACK copy of a CSR matrix that the CG mat-vec reads (system.h).
 * First call with sellCol == NULL to get the padded entry count in *paddedNnz; sellPtr holds (n + 31) / 32 + 1
 * words, sellRow 32 per slice (0xffffffff = padding lane).  Replaces nothing in the reference (its LLT reads
 * Eigen's CSC, Solver.cpp:213-215); exposed so the layout is testable without a GPU. */
int pies_b200_probe_sell(uint32_t n, const int32_t* rowPtr, const int32_t* col, const float* val, uint32_t* sellPtr,
                         uint32_t* sellRow, int32_t* sellCol, float* sellVal, uint64_t* paddedNnz);

/* Host only: the closed segments of the fused local step + RHS (one CTA per segment, see DESIGN.md section 4) of a
 * scene built from nCmds commands of 8 floats (kind, tx, ty, tz, a, b, c, d), t = translation:
 *   kind 0: createTetBox(t, scale a, v0 0, w b, mass c, not hinged)
 *   kind 1: createSheet(t, scale a, mass b, k c)
 *   kind 2: createShapeMatchingBox(t, a x b x c particles, scale d, v0 0, w 1000)
 *   kind 3: addTetMeshVolume of meshPoints + t and meshTets (no triangles), density 1, strain w 1000 in [0.8, 1],
 *           volume w 1000 in [1, 1]
 * sizes[0..6] = nodes, gather-list entries, fused tet elements, segments, elements outside segments, nodes outside
 * segments, first tet contribution slot.  The arrays may be null (first call: sizes only); otherwise incPtr (nodes + 1),
 * inc and segSlot (entries), elemIds (4 per element), segs (4 per segment: n0, n1, e0, e1), restElems, restNodes. */
int pies_b200_probe_segments(uint32_t nCmds, const float* cmds, uint32_t nMeshPoints, const float* meshPoints,
                             uint32_t nMeshTets, const uint32_t* meshTets, uint64_t* sizes, int32_t* incPtr, uint32_t* inc,
                             uint16_t* segSlot, uint32_t* elemIds, uint32_t* segs, uint32_t* restElems,
                             uint32_t* restNodes);

#ifdef __cplusplus
}
#endif
#endif /* PIES_B200_H */
