// engine.h — the solver object behind the C ABI: host scene + device state + tick loops.
#pragma once

#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "kernels.h"
#include "scene.h"
#include "system.h"

namespace pies {

// Stream every grow-only buffer (re)allocates on: the calling solver's stream, set at each C-ABI entry
// (capi.cpp: guarded()).  Allocation is stream-ordered (cudaMallocAsync from the device's default pool, whose
// release threshold pies_b200_create raises so freed blocks stay cached): growing a contact-sized buffer in
// the middle of a substep neither synchronises the device nor goes back to the driver for memory.
inline thread_local cudaStream_t g_allocStream = nullptr;

template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;
  ~DevBuf() { release(); }
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }  // synchronising; destructor / clear only
  // grow-only; contents are NOT preserved.  Work already enqueued on the stream keeps the old block (the free is stream-ordered).
  cudaError_t reserve(size_t n) {
    if (n <= cap) return cudaSuccess;
    if (p) { cudaFreeAsync(p, g_allocStream); p = nullptr; cap = 0; }
    size_t want = 2 * n + 64;  // geometric growth: contact-sized buffers grow a little every substep
    cudaError_t e = cudaMallocAsync(reinterpret_cast<void**>(&p), want * sizeof(T), g_allocStream);
    if (e == cudaSuccess) cap = want; else p = nullptr;
    return e;
  }
  cudaError_t upload(const T* src, size_t n, cudaStream_t s) {
    cudaError_t e = reserve(n);
    if (e != cudaSuccess || !n) return e;
    return cudaMemcpyAsync(p, src, n * sizeof(T), cudaMemcpyHostToDevice, s);
  }
};

struct DetectWork;   // detect.cu
struct ContactWork;  // contact.cu
struct BlockWork;    // reblock.cu
struct IslandWork;   // islands.cu
struct HaloWork;     // halo.cu
struct PbdWork;      // pbd.cu
void destroyPbdWork(PbdWork* w);

}  // namespace pies

struct PiesB200Solver {
  pies::HostScene scene;
  PiesB200Options opt{};
  PiesB200Tuning tune{};
  PiesB200Stats stats{};
  bool releaseHinge = false, renderStateDirty = true, simFailed = false;
  std::string err;

  int device = 0;
  cudaStream_t stream = nullptr;
  bool ownStream = false;

  // ---- device state ----
  uint64_t builtVersion = ~0ull;
  bool deviceNewer = false;   // device q/prev/vel are ahead of scene.pos/prev/vel
  bool mirrorStale = false;     // scene.vertices[].position is behind the device; refreshed lazily by get_vertices
  bool hostStateDirty = false; // scene.pos/prev/vel were overwritten (set_state) and must be re-uploaded
  uint32_t n = 0;
  pies::HostSystem sys;
  pies::DevBuf<float4> q, prev, vel, msn, rhs, contrib, snap;
  pies::DevBuf<float4> pr, pp, pp2, pz, pap, pdelta;
  pies::DevBuf<float> partials, scalars;
  pies::DevBuf<int> flag;
  pies::DevBuf<uint4> elemIds;
  pies::DevBuf<float4> elemQa, elemQb, elemPc, elemPd, elemRot;
  pies::DevBuf<uint2> distIds; pies::DevBuf<float2> distRestW;
  pies::DevBuf<uint4> bendIds; pies::DevBuf<float2> bendAngleW;
  pies::DevBuf<uint32_t> shapeOff, shapeIds, goalOff, goalIds;
  pies::DevBuf<double> shapeMat, shapeQinv, shapeQuat;
  pies::DevBuf<float> shapeW, goalMat, goalXform, goalW;
  pies::DevBuf<int> incPtr; pies::DevBuf<uint32_t> inc;
  pies::DevBuf<uint4> segs; pies::DevBuf<uint16_t> segSlot; pies::DevBuf<uint32_t> restElems, restNodes;  // HostSystem::segs
  pies::DevBuf<int> rowPtr, col; pies::DevBuf<float> val;
  pies::DevBuf<uint32_t> sellPtr, sellRow; pies::DevBuf<int> sellCol; pies::DevBuf<float> sellVal;
  pies::DevBuf<int> blockNodes; pies::DevBuf<float> blockInv;
  pies::DevBuf<uint32_t> triIds;  // 3 per triangle
  pies::DevBuf<float> packed;     // 3 floats per node, readback staging
  // Device-side copy of the Vertex mirror (36 B per vertex, Solver.h:42-49): the static attributes are uploaded once per
  // topology, a kernel refreshes the positions, and getVertices() is one contiguous DMA into the (page-locked) host vector.
  pies::DevBuf<float> vtxDev; bool vtxDevValid = false;
  float* vtxExternal = nullptr;   // caller-owned device vertex buffer (render interop), used instead of vtxDev when set
  void* vtxRegistered = nullptr; size_t vtxRegisteredBytes = 0;  // the host vector's storage while it is cudaHostRegister-ed
  // PBD
  pies::DevBuf<uint32_t> posIds; pies::DevBuf<float4> posTargetW;

  pies::DetectWork* detect = nullptr;
  pies::ContactWork* contact = nullptr;
  pies::BlockWork* blocks = nullptr;
  pies::IslandWork* islands = nullptr;
  pies::HaloWork* halo = nullptr;   // set by pies_b200_halo_init: slab-partitioned multi-GPU run
  pies::PbdWork* pbd = nullptr;
  void* pdCtx = nullptr;          // PdTickCtx of a tick in progress (engine.cu)
  pies::DevBuf<uint32_t> triOrder; bool haveTriOrder = false;  // canonical-order override (slab-partitioned hosts)
  pies::DevBuf<uint32_t> ownedCount;  // output of countOwnedContacts (its own buffer: `flag` belongs to the CG reductions)
  pies::DevBuf<uint8_t> ownedMask; bool haveOwnedMask = false; // nodes this rank owns (others are ghosts)
  // static colliders (colliders.cu): the validated set, its device copy, the per-node contact masks of the last detection
  // (valid for colMaskColliders colliders; 0 = none) and the per-iteration sum of their weighted projections
  std::vector<PiesB200Collider> colliderSet;
  pies::DevBuf<PiesB200Collider> colliders;
  pies::DevBuf<uint32_t> colMask; pies::DevBuf<float4> colRhs;
  uint32_t colMaskColliders = 0;
  // drag targets (pick.cu): the validated set's size and its device copy (node ids, (g, w)); dragCount = 0 = none
  uint32_t dragCount = 0;
  pies::DevBuf<uint32_t> dragNode; pies::DevBuf<float4> dragTargetW;
  // external forces (forces.cu): the validated host set (copied by set_external_forces; uploaded as the dense per-node
  // buffer hostForce, zeros for unlisted nodes, at the first tick after a change or a node-count change), the wind
  // (wind = (velocity, c_n), windTangential = c_t; both coefficients 0 = none) with its node -> triangle CSR of topology
  // windCsrVersion, per-triangle slots and per-node sums (allocated at the first tick with wind), and what the last tick
  // applied: forceMode bit 1 = hostForce, bit 2 = wind (fext), for forceModeN nodes
  std::vector<uint32_t> forceIds; std::vector<float4> forceVals;
  bool forceDirty = false; uint32_t forceDenseN = 0;
  pies::DevBuf<float4> hostForce;
  float4 wind{0.0f, 0.0f, 0.0f, 0.0f}; float windTangential = 0.0f;
  uint64_t windCsrVersion = ~0ull;
  pies::DevBuf<int> windPtr; pies::DevBuf<uint32_t> windList; pies::DevBuf<float4> windSlot, fext;
  uint32_t forceMode = 0, forceModeN = 0;
  // raycast staging (pick.cu): rays (2 float4 each), per-ray hit keys, packed results
  pies::DevBuf<float4> rays; pies::DevBuf<unsigned long long> rayKey; pies::DevBuf<float4> rayHit;

  float* hostPacked = nullptr;  // pinned, 3 floats per node
  size_t hostPackedCap = 0;
  int* hostFlag = nullptr;      // pinned, 4 ints
  uint32_t lastPcgIters = 1;
  std::vector<cudaEvent_t> eventPool;  // phase-timing events of this solver (created on its device)
  cudaEvent_t tickEv[2] = {nullptr, nullptr};  // brackets of the whole tick, created once
  std::vector<uint32_t> pcgItersByIteration;  // CG iterations the k-th PD iteration of the previous substep needed (burst prediction)
  uint64_t launches = 0;

  ~PiesB200Solver();
};

namespace pies {
int failCuda(PiesB200Solver* s, cudaError_t e, const char* what, int line);
int ensureTickEvents(PiesB200Solver* s);
int fail(PiesB200Solver* s, int code, const char* msg);
int ensureBuilt(PiesB200Solver* s);
int downloadState(PiesB200Solver* s);  // device -> scene.pos/prev/vel
int downloadVec3(PiesB200Solver* s, const float4* src, float* dstXYZ);  // one device plane -> packed xyz in the caller's (pinned or pageable) buffer
int tickPD(PiesB200Solver* s, bool refreshMirror);
int pdTickBegin(PiesB200Solver* s);
int pdSubstepBegin(PiesB200Solver* s);
int pdIteration(PiesB200Solver* s);
int pdSubstepEnd(PiesB200Solver* s);
int pdTickEnd(PiesB200Solver* s, bool refreshMirror);
void pdAbort(PiesB200Solver* s);
int countOwnedContacts(PiesB200Solver* s, uint32_t* nTri, uint32_t* nFloor);
int tickPBD(PiesB200Solver* s, bool refreshMirror);
int refreshVertexMirror(PiesB200Solver* s);
int refreshDeviceVertices(PiesB200Solver* s, float** out);  // positions into the device-side Vertex array, no host copy
void unregisterVertexMirror(PiesB200Solver* s);  // before anything that may reallocate scene.vertices
int uploadStateArrays(PiesB200Solver* s, const float* pos, const float* prev, const float* vel);
int runDetection(PiesB200Solver* s, ContactLists& lists);
int pbdHashOnly(PiesB200Solver* s);
// Checks a caller's collider set (include/pies_b200.h: set_colliders) into out, half-space normals normalised; on failure
// returns PIES_B200_EINVAL / ERANGE with the reason in *why.
int prepareColliders(uint32_t n, const PiesB200Collider* in, std::vector<PiesB200Collider>& out, const char** why);
int setColliders(PiesB200Solver* s, uint32_t n, const PiesB200Collider* c);
inline ColliderSet colliderSet(const PiesB200Solver* s) { return ColliderSet{s->colliders.p, (uint32_t)s->colliderSet.size()}; }
int setDragTargets(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* targets, const float* weights);
inline DragSet dragSet(const PiesB200Solver* s) { return DragSet{s->dragNode.p, s->dragTargetW.p, s->dragCount}; }
int setExternalForces(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* forces);
int setWind(PiesB200Solver* s, const float* velocity, float normalDrag, float tangentialDrag);
int prepareForces(PiesB200Solver* s);   // tick start, after ensureBuilt
int getExternalForces(PiesB200Solver* s, float* xyz);
void clearForces(PiesB200Solver* s);
// the forces the current (or last) tick applies, as fixed by prepareForces
inline ForceSet forceSet(const PiesB200Solver* s) {
  ForceSet f;
  if (s->forceMode & 1u) f.host = s->hostForce.p;
  if (s->forceMode & 2u) {
    f.nTri = s->scene.triCount(); f.tri = s->triIds.p; f.ptr = s->windPtr.p; f.list = s->windList.p;
    f.slot = s->windSlot.p; f.fext = s->fext.p; f.wind = s->wind; f.ct = s->windTangential;
  }
  return f;
}
int raycast(PiesB200Solver* s, uint32_t nRays, const float* origins, const float* dirs, const float* tMax, int32_t* tri,
            float* t, float* uv);
int pbdOccupancyCounts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers);
int pbdOccupancy(PiesB200Solver* s, int64_t* cellsXYZ, uint32_t* counts, uint32_t* members);
}  // namespace pies

#define PIES_CHECK(s, expr)                                                        \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) return pies::failCuda((s), _e, #expr, __LINE__);        \
  } while (0)
