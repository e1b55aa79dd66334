// kernels.h — launch wrappers of the sm_100a kernels (host-callable).
// Every wrapper enqueues on the given stream and returns the number of kernel
// launches it made (so the engine can report gpu_launches honestly).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/pies_b200.h"

namespace pies {

// ---------------------------------------------------------------- layouts ----
// Node state, one float4 per node so a constraint gathers a node with one 16 B load:
//   q    = (x, y, z, invMass)         current position
//   prev = (x, y, z, radius)          Node::prevPosition
//   vel  = (vx, vy, vz, 0)
//   msn  = M s_n / h^2 (Solver.cpp:234-237), rhs = right-hand side of the global step.
//
// Fused tet elements: a strain constraint and a volume constraint on the same tet share
// ids and Qinv, so they are stored (and their SVD computed) once.  Five 16 B planes:
struct TetElems {
  uint4* ids = nullptr;      // node ids
  float4* qa = nullptr;      // Qinv[0..3]   (glm column-major)
  float4* qb = nullptr;      // Qinv[4..7]
  float4* pc = nullptr;      // Qinv[8], wStrain, minStrain, maxStrain
  float4* pd = nullptr;      // wVolume, minOmega, maxOmega, unused
  float4* rot = nullptr;     // state: 2 unit quaternions per tet (U, V of the last SVD), warm start of the next; null = cold start
  uint32_t n = 0;
};

// Closed segments of the fused local step + RHS (k_tet_rhs; built by buildSegments, system.h): per segment the node
// range [n0, n1) and the element range [e0, e1) that one CTA projects and assembles on chip.
constexpr uint32_t kSegElems = 256;     // cap per segment: 4 float4 contributions per element in shared memory ...
constexpr uint32_t kSegNodes = 256;     // ... and one staged float4 position per node (20 KB per CTA)
constexpr int kTetRhsThreads = 128;     // CTA of k_tet_rhs (elements, then nodes, strided over the threads)
struct TetSegments {
  const uint4* segs = nullptr;          // (n0, n1, e0, e1)
  const uint16_t* slot = nullptr;       // parallel to the gather list inc: 4 (e - e0) + k for the nodes of a segment
  uint32_t n = 0;
};

struct DistanceElems { uint2* ids = nullptr; float2* restW = nullptr; uint32_t n = 0; };
struct BendElems { uint4* ids = nullptr; float2* angleW = nullptr; uint32_t n = 0; };
struct ClusterElems {  // shape- and goal-matching clusters (CSR over members)
  uint32_t* off = nullptr;   // nClusters + 1
  uint32_t* ids = nullptr;   // member node ids
  uint32_t nClusters = 0, nMembers = 0;
};

// CSR of S = M/h^2 + sum w A^T A (Solver.cpp:174-210), both triangles.
struct CsrMatrix {
  int* rowPtr = nullptr; int* col = nullptr; float* val = nullptr; uint32_t n = 0; uint64_t nnz = 0;
  // sliced-ELLPACK copy read by the CG mat-vec (system.h): slice s holds rows sellRow[32 s + lane], entry k of a
  // lane at sellPtr[s] + 32 k + lane
  uint32_t* sellPtr = nullptr; uint32_t* sellRow = nullptr; int* sellCol = nullptr; float* sellVal = nullptr;
  uint32_t nSlices = 0;
  uint64_t sellEntries = 0;  // padded entries of the SELL copy (picks the mat-vec's tile variant)
};

// Per-substep collision lists in the reference's canonical order.
struct ContactLists {
  uint4* tri = nullptr;        // (a, b, c, d): point a against triangle (b, c, d)
  uint32_t* floorNode = nullptr;
  uint32_t nTri = 0, nFloor = 0;
  // distinct (point, triangle) contacts with their weight = copies * 1e4 (the list above holds one copy
  // per shared cell, SURVEY F7): what the collision matrix and the right-hand side are built from
  uint4* uTri = nullptr; float* uW = nullptr; uint32_t nUnique = 0;
  // node -> incident distinct contacts, CSR (value = 4 * contact + slot), contacts ascending
  int* incPtr = nullptr; uint32_t* inc = nullptr;
  float* floorW = nullptr;     // per node: sum of floor-contact weights (multiplicity * 1e4)
  // The same collision matrix C_t in streamable form (what the CG mat-vec reads): off-diagonal entries as CSR
  // (a point row holds -w for its three triangle corners, a corner row -w for the point; entries in incidence
  // order) and the per-node diagonal sum (3 w / w per contact + the floor and collider weights).  cDiag is valid
  // when nTri || nodeWeights(), the CSR when nUnique.
  int* cPtr = nullptr; int* cCol = nullptr; float* cVal = nullptr; float* cDiag = nullptr;
  uint32_t* floorMult = nullptr;
  // ordered Gauss-Seidel sweeps: ticket[e] = position of entry e in each of its four nodes' incidence
  // lists; nodeDone[v] = entries touching v already executed in the current sweep
  uint4* ticket = nullptr;
  uint32_t* nodeDone = nullptr;
  // Static colliders (colliders.cu): the solver's collider count when this detection wrote colMask, else 0.  A host count,
  // not a contact count, so nothing is read back.  When it is set, floorW and cDiag also hold 1e4 per mask bit.
  uint32_t nCollide = 0;
  // Drag targets (pick.cu): the solver's drag count when this detection added their weights to floorW and cDiag (and
  // w g to msn), else 0.  Also a host count; it fills the padding before colMask, so the struct keeps its size.
  uint32_t nDrag = 0;
  const uint32_t* colMask = nullptr;   // per node: bit k = in contact with collider k
  const float4* colRhs = nullptr;      // per node with a mask: sum over its bits (ascending) of 1e4 p_k, this PD iteration
  // floorW / cDiag carry one-node weights (floor, collider or drag)
  __host__ __device__ bool nodeWeights() const { return nFloor || nCollide || nDrag; }
};

// ------------------------------------------------------------- PD kernels ----
int launchPredict(cudaStream_t s, uint32_t n, float4* q, const float4* vel, float4* msn, float h);
// list: the n elements to project (null = 0 .. n-1)
int launchTetElems(cudaStream_t s, const TetElems& e, const uint32_t* list, uint32_t n, const float4* q, float4* contrib);
int launchDistance(cudaStream_t s, const DistanceElems& e, const float4* q, float4* contrib);
int launchBend(cudaStream_t s, const BendElems& e, const float4* q, float4* contrib);
int launchGoal(cudaStream_t s, const ClusterElems& c, const float* material /*3 per member*/,
               const float* xform /*16 per cluster*/, const float* w, float4* contrib);
int launchShape(cudaStream_t s, const ClusterElems& c, const double* material, const double* qinv,
                double* quat /*4 per cluster, state*/, const float* w, const float4* q, float4* contrib);
// nodes: the n nodes to assemble (null = 0 .. n-1)
int launchGatherRhs(cudaStream_t s, uint32_t n, const uint32_t* nodes, const float4* msn, const int* incPtr,
                    const uint32_t* inc, const float4* contrib, float4* rhs);
// Fused tet projections + RHS of every node of the segments (with the collision and floor terms of c when it has any).
int launchTetRhs(cudaStream_t s, const TetElems& e, const TetSegments& sg, const float4* q, const float4* msn,
                 const int* incPtr, const ContactLists& c, const float4* contribC, float4* snap, float4* rhs);
// fext: per-node external force (ForceSet::field()), null = none: the parent's k_velocity
int launchVelocityUpdate(cudaStream_t s, uint32_t n, const float4* q, float4* prev, float4* vel, float h,
                         float damping, float gravity, const float4* fext);

// ------------------------------------------------------ static colliders -----
// (colliders.cu; col = the solver's device copy of its colliders, n of them)
struct ColliderSet { const PiesB200Collider* col = nullptr; uint32_t n = 0; };
// Detection: mask of every node (phi_k(q) < thickness), and floorW[i] = (haveFloor ? floorW[i] : 0) + 1e4 per mask bit.
int launchColliderDetect(cudaStream_t s, uint32_t n, const ColliderSet& c, const float4* q, float thickness,
                         bool haveFloor, uint32_t* mask, float* floorW);
// Local step: colRhs[i] = sum over the mask bits of node i (ascending) of 1e4 p_k(q_i).
int launchColliderProject(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, const float4* q,
                          float4* colRhs);
// After stabilisation: q of every node with a mask projected through its colliders in sequence.
int launchColliderSnap(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, float4* q);
// After the floor friction: the friction rule of k_floor_friction in each contact's tangent plane.
int launchColliderFriction(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, const float4* q,
                           float4* vel, float friction, float staticThreshold);
// PBD: after the floor clamp / after the velocity update (radius = prev.w).
int launchPbdColliderClamp(cudaStream_t s, uint32_t n, const ColliderSet& c, float4* q, const float4* prev);
int launchPbdColliderFriction(cudaStream_t s, uint32_t n, const ColliderSet& c, const float4* q, const float4* prev,
                              float4* vel, float friction);
void preloadColliderKernels();

// ---------------------------------------------------------- drag targets -----
// (pick.cu; node[k] with targetW[k] = (g, w), ids unique)
struct DragSet { const uint32_t* node = nullptr; const float4* targetW = nullptr; uint32_t n = 0; };
// PD detection, after the floor and collider weights: floorW[node] += w, msn[node] += w g.
int launchDragTerms(cudaStream_t s, const DragSet& d, float* floorW, float4* msn);
// PBD, after the position-constraint sweep: x += min(w, 1) (g - x).
int launchPbdDrag(cudaStream_t s, const DragSet& d, float4* q);

// ------------------------------------------------------- external forces -----
// (forces.cu) host: dense per-node host forces, or null.  nTri > 0: wind on the triangles tri (3 ids each) with
// wind = (w, c_n) and c_t = ct, over the node -> triangle CSR (ptr, list), one slot per triangle, summed into fext.
struct ForceSet {
  const float4* host = nullptr;
  uint32_t nTri = 0;
  const uint32_t* tri = nullptr; const int* ptr = nullptr; const uint32_t* list = nullptr;
  float4* slot = nullptr; float4* fext = nullptr;
  float4 wind{0.0f, 0.0f, 0.0f, 0.0f}; float ct = 0.0f;
  // what the velocity update (PD) or the advection (PBD) reads: null = no external force
  const float4* field() const { return nTri ? fext : host; }
};
// Substep start, before k_predict / k_pbd_advect: k_wind_tri + k_force_gather into fext when nTri > 0, else nothing.
int launchForces(cudaStream_t s, uint32_t n, const ForceSet& f, const float4* q, const float4* vel);

// ------------------------------------------------------------------ PCG -----
struct PcgWork {
  float4 *r = nullptr, *p = nullptr, *p2 = nullptr, *z = nullptr, *ap = nullptr, *delta = nullptr;
  float* partials = nullptr;   // kMaxReduceBlocks * 32 floats (per-CTA partial sums, kPartialStride apart)
  float* scalars = nullptr;    // see pcg.cu
  int* flag = nullptr;         // [0] converged, [1] iterations done, [2] ticket counter of the grid reductions
  // block-Jacobi preconditioner (rebuilt per substep, reblock.cu): blocks of m <= 32 nodes, dense inverse of
  // S + C_t restricted to the block
  int* blockNodes = nullptr;   // nBlocks * 32 node ids, members first (-1 = padding)
  float* blockInv = nullptr;   // per block: packed lower triangle of the symmetric m x m inverse, (j, i <= j) at j (j + 1) / 2 + i
  const uint2* blockMeta = nullptr;        // per block: (offset into blockInv in floats, m)
  uint32_t nBlocks = 0;                    // upper bound used for grid sizing
  const uint32_t* nBlocksDev = nullptr;    // actual block count of this substep (device)
  // Restriction of the grid-wide solve to the islands the island-local kernels left over (islands.cu); all null = every
  // row.  big[i] != 0: node i takes part; actWin: ascending list of the 256-row windows holding such a node, actBlk: of
  // the preconditioner blocks made of such nodes; counts[0] = #windows, counts[1] = #blocks (device).
  const uint8_t* big = nullptr;
  const uint32_t* actWin = nullptr;
  const uint32_t* actBlk = nullptr;
  const uint32_t* actCounts = nullptr;
};
// Solves A (x + delta) = b for the correction delta, starting from delta = 0 with the start
// residual b - A x accumulated in fp64.
int launchPcgInit(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w,
                  const float4* b, const float4* x, float tol);
// it = iteration index within the solve (parity selects the double-buffered r.z slot and direction buffer)
int launchPcgIteration(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w, float tol, int it);
int launchPcgSpmv(cudaStream_t s, const CsrMatrix& A, const ContactLists& c, const PcgWork& w, float tol, int it);  // first half of an iteration
int launchPcgUpdate(cudaStream_t s, const PcgWork& w, float tol, int it);                                          // second half
int launchPcgCheck(cudaStream_t s, const PcgWork& w, float tol, int lastIt);
// x += delta: the correction is accumulated separately and added with a single rounding
int launchPcgFinish(cudaStream_t s, const PcgWork& w, uint32_t n, float4* x);

// ----------------------------------------------------------------- scan -----
// In-place exclusive scan of data[0..n); scratch holds scanScratchElems(n) uint32.
size_t scanScratchElems(uint64_t n);
int launchExclusiveScan(cudaStream_t s, uint32_t* data, uint64_t n, uint32_t* scratch);

// ----------------------------------------------------------------- sort -----
// Stable LSD radix sort of (64-bit key, 32-bit value) pairs on keyBits low bits.
// keys/vals are sorted in place; tmpKeys/tmpVals are same-size scratch; hist is
// scratch of sortHistBytes(n) bytes.
size_t sortHistBytes(uint64_t n);
int launchSortPairs(cudaStream_t s, uint64_t n, uint64_t* keys, uint32_t* vals, uint64_t* tmpKeys,
                    uint32_t* tmpVals, void* hist, int keyBits);

// ------------------------------------------------------------- preload -----
// Force-load every kernel of a file (no lazy loading in the middle of a run).
void preloadDetectKernels();
void preloadContactKernels();
void preloadReblockKernels();
void preloadSortKernels();
void preloadPcgKernels();

}  // namespace pies
