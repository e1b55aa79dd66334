// engine.cu — device-state management and the per-timestep loops of the B200 solver.
//
// tickPD follows reference Solver::tickPD (Src/Solver.cpp:162-486) phase by phase; each
// phase is one or a few kernels on the solver's stream.  There is no CPU path: if CUDA
// fails the solver latches simFailed (the reference's only failure mode, Solver.cpp:26-28)
// and reports the error.
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <thread>

#include "common.cuh"
#include "contact.h"
#include "detect.h"
#include "halo.h"
#include "islands.h"
#include "reblock.h"

namespace pies {

int fail(PiesB200Solver* s, int code, const char* msg) {
  if (s) s->err = msg;
  return code;
}

int failCuda(PiesB200Solver* s, cudaError_t e, const char* what, int line) {
  char buf[512];
  std::snprintf(buf, sizeof(buf), "CUDA error %d (%s) at engine.cu:%d: %s", (int)e, cudaGetErrorString(e), line, what);
  if (s) { s->err = buf; s->simFailed = true; }
  return PIES_B200_ECUDA;
}

// pack kernel for the readback path: float4 (x,y,z,*) -> 3 contiguous floats
__global__ void __launch_bounds__(kThreads) k_pack3(uint32_t n, const float4* __restrict__ src, float* __restrict__ dst) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 v = src[i];
  dst[3ull * i] = v.x; dst[3ull * i + 1] = v.y; dst[3ull * i + 2] = v.z;
}

// inverse of k_pack3 for the set_state path; keeps .w (invMass / radius)
__global__ void __launch_bounds__(kThreads) k_unpack3(uint32_t n, const float* __restrict__ src, float4* __restrict__ dst) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 v = dst[i];
  v.x = src[3ull * i]; v.y = src[3ull * i + 1]; v.z = src[3ull * i + 2];
  dst[i] = v;
}

static int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

template <typename T, typename U>
static cudaError_t uploadVec(DevBuf<T>& d, const std::vector<U>& h, cudaStream_t s) {
  static_assert(sizeof(T) % sizeof(U) == 0, "element packing");
  return d.upload(reinterpret_cast<const T*>(h.data()), h.size() * sizeof(U) / sizeof(T), s);
}

int ensureTickEvents(PiesB200Solver* s) {
  for (int k = 0; k < 2; ++k)
    if (!s->tickEv[k]) PIES_CHECK(s, cudaEventCreate(&s->tickEv[k]));
  return PIES_B200_OK;
}

int downloadVec3(PiesB200Solver* s, const float4* src, float* dstXYZ) {
  uint32_t n = s->n;
  if (!n) return PIES_B200_OK;
  PIES_CHECK(s, s->packed.reserve(3ull * n));
  if (s->hostPackedCap < 3ull * n) {
    if (s->hostPacked) cudaFreeHost(s->hostPacked);
    s->hostPacked = nullptr; s->hostPackedCap = 0;
    PIES_CHECK(s, cudaMallocHost(&s->hostPacked, (3ull * n + 64) * sizeof(float)));
    s->hostPackedCap = 3ull * n + 64;
  }
  k_pack3<<<gridFor(n, kThreads), kThreads, 0, s->stream>>>(n, src, s->packed.p);
  ++s->launches;
  // A page-locked destination takes the DMA directly; pageable memory goes through the solver's pinned staging buffer.
  cudaPointerAttributes attr{};
  const bool pinned = cudaPointerGetAttributes(&attr, dstXYZ) == cudaSuccess && attr.type == cudaMemoryTypeHost;
  if (!pinned) cudaGetLastError();
  float* dmaDst = pinned ? dstXYZ : s->hostPacked;
  PIES_CHECK(s, cudaMemcpyAsync(dmaDst, s->packed.p, 3ull * n * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  if (!pinned) std::memcpy(dstXYZ, s->hostPacked, 3ull * n * sizeof(float));
  return PIES_B200_OK;
}

// Host arrays (pinned or pageable) -> device state, without touching the topology.
int uploadStateArrays(PiesB200Solver* s, const float* pos, const float* prev, const float* vel) {
  uint32_t n = s->n;
  if (!n) return PIES_B200_OK;
  PIES_CHECK(s, s->packed.reserve(9ull * n));
  const float* src[3] = {pos, prev, vel};
  float4* dst[3] = {s->q.p, s->prev.p, s->vel.p};
  for (int k = 0; k < 3; ++k) {
    if (!src[k]) continue;
    float* stage = s->packed.p + 3ull * n * k;
    PIES_CHECK(s, cudaMemcpyAsync(stage, src[k], 3ull * n * sizeof(float), cudaMemcpyHostToDevice, s->stream));
    k_unpack3<<<gridFor(n, kThreads), kThreads, 0, s->stream>>>(n, stage, dst[k]);
    ++s->launches;
  }
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  s->deviceNewer = true;
  return PIES_B200_OK;
}

int downloadState(PiesB200Solver* s) {
  if (!s->deviceNewer || !s->n) { s->deviceNewer = false; return PIES_B200_OK; }
  int rc;
  if ((rc = downloadVec3(s, s->q.p, s->scene.pos.data()))) return rc;
  if ((rc = downloadVec3(s, s->prev.p, s->scene.prev.data()))) return rc;
  if ((rc = downloadVec3(s, s->vel.p, s->scene.vel.data()))) return rc;
  if (s->scene.shapeQuat.size() && s->shapeQuat.p)
    PIES_CHECK(s, cudaMemcpy(s->scene.shapeQuat.data(), s->shapeQuat.p,
                             std::min(s->scene.shapeQuat.size(), s->shapeQuat.cap) * sizeof(double), cudaMemcpyDeviceToHost));
  s->deviceNewer = false;
  return PIES_B200_OK;
}

static int uploadState(PiesB200Solver* s) {
  const HostScene& sc = s->scene;
  uint32_t n = sc.nodeCount();
  std::vector<float4> q(n), pv(n), vl(n);
  for (uint32_t i = 0; i < n; ++i) {
    q[i] = make_float4(sc.pos[3 * i], sc.pos[3 * i + 1], sc.pos[3 * i + 2], sc.invMass[i]);
    pv[i] = make_float4(sc.prev[3 * i], sc.prev[3 * i + 1], sc.prev[3 * i + 2], sc.radius[i]);
    vl[i] = make_float4(sc.vel[3 * i], sc.vel[3 * i + 1], sc.vel[3 * i + 2], 0.0f);
  }
  PIES_CHECK(s, s->q.upload(q.data(), n, s->stream));
  PIES_CHECK(s, s->prev.upload(pv.data(), n, s->stream));
  PIES_CHECK(s, s->vel.upload(vl.data(), n, s->stream));
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));  // staging vectors die here
  return PIES_B200_OK;
}

// Rebuild the device-side topology when the scene changed.  The reference rebuilds only when
// the NODE count changes (Solver.cpp:168-169, SURVEY F2 — constraints added later never reach
// its system matrix); here any scene mutation triggers the rebuild, which is identical for hosts
// that add whole bodies and strictly safer otherwise.
int ensureBuilt(PiesB200Solver* s) {
  HostScene& sc = s->scene;
  if (s->builtVersion == sc.topologyVersion) {
    if (s->hostStateDirty) {
      int rcu = uploadState(s);
      if (rcu) return rcu;
      s->hostStateDirty = false;
    }
    if (sc.goalXformDirty && sc.goalXform.size()) {
      PIES_CHECK(s, s->goalXform.upload(reinterpret_cast<const float*>(sc.goalXform.data()), sc.goalXform.size() * 16, s->stream));
      PIES_CHECK(s, cudaStreamSynchronize(s->stream));
      sc.goalXformDirty = false;
    }
    return PIES_B200_OK;
  }
  int rc = downloadState(s);
  if (rc) return rc;
  const uint32_t n = sc.nodeCount();
  s->n = n;
  float h = s->opt.fixedTimestepSize / (float)s->opt.timeSubsteps;
  unsigned hw = std::max(1u, std::min(16u, std::thread::hardware_concurrency()));
  buildSystem(sc, h, s->sys, hw);
  const HostSystem& y = s->sys;
  cudaStream_t st = s->stream;
  if ((rc = uploadState(s))) return rc;
  PIES_CHECK(s, s->msn.reserve(n)); PIES_CHECK(s, s->rhs.reserve(n)); PIES_CHECK(s, s->snap.reserve(n));
  PIES_CHECK(s, s->pr.reserve(n)); PIES_CHECK(s, s->pp.reserve(n)); PIES_CHECK(s, s->pp2.reserve(n)); PIES_CHECK(s, s->pz.reserve(n)); PIES_CHECK(s, s->pap.reserve(n)); PIES_CHECK(s, s->pdelta.reserve(n));
  PIES_CHECK(s, s->partials.reserve((size_t)kMaxReduceBlocks * 32)); PIES_CHECK(s, s->scalars.reserve(64)); PIES_CHECK(s, s->flag.reserve(4));
  PIES_CHECK(s, cudaMemsetAsync(s->partials.p, 0, (size_t)kMaxReduceBlocks * 32 * sizeof(float), st));
  PIES_CHECK(s, cudaMemsetAsync(s->scalars.p, 0, 64 * sizeof(float), st));
  PIES_CHECK(s, cudaMemsetAsync(s->flag.p, 0, 4 * sizeof(int), st));
  PIES_CHECK(s, cudaMemsetAsync(s->snap.p, 0, (size_t)n * sizeof(float4), st));
  PIES_CHECK(s, s->contrib.reserve(y.nContrib + 1));
  PIES_CHECK(s, cudaMemsetAsync(s->contrib.p, 0, (y.nContrib + 1) * sizeof(float4), st));
  if (y.posContrib.size())
    PIES_CHECK(s, cudaMemcpyAsync(s->contrib.p + y.basePos, y.posContrib.data(), y.posContrib.size() * sizeof(float),
                                  cudaMemcpyHostToDevice, st));
  PIES_CHECK(s, uploadVec(s->elemIds, y.elemIds, st));
  PIES_CHECK(s, uploadVec(s->elemQa, y.elemQa, st)); PIES_CHECK(s, uploadVec(s->elemQb, y.elemQb, st));
  PIES_CHECK(s, uploadVec(s->elemPc, y.elemPc, st)); PIES_CHECK(s, uploadVec(s->elemPd, y.elemPd, st));
  {  // SVD warm-start state: identity rotations
    std::vector<float4> ident(2ull * y.nElems, make_float4(0.0f, 0.0f, 0.0f, 1.0f));
    PIES_CHECK(s, s->elemRot.upload(ident.data(), ident.size(), st));
    PIES_CHECK(s, cudaStreamSynchronize(st));
  }
  PIES_CHECK(s, uploadVec(s->distIds, sc.distId, st));
  {
    std::vector<float2> rw(sc.distW.size());
    for (size_t i = 0; i < rw.size(); ++i) rw[i] = make_float2(sc.distRest[i], sc.distW[i]);
    PIES_CHECK(s, s->distRestW.upload(rw.data(), rw.size(), st));
    std::vector<float2> aw(sc.bendW.size());
    for (size_t i = 0; i < aw.size(); ++i) aw[i] = make_float2(sc.bendAngle[i], sc.bendW[i]);
    PIES_CHECK(s, s->bendAngleW.upload(aw.data(), aw.size(), st));
    std::vector<float4> pt(sc.posW.size());
    for (size_t i = 0; i < pt.size(); ++i) pt[i] = make_float4(sc.posTarget[3 * i], sc.posTarget[3 * i + 1], sc.posTarget[3 * i + 2], sc.posW[i]);
    PIES_CHECK(s, s->posTargetW.upload(pt.data(), pt.size(), st));
    PIES_CHECK(s, cudaStreamSynchronize(st));
  }
  PIES_CHECK(s, uploadVec(s->posIds, sc.posId, st));
  PIES_CHECK(s, uploadVec(s->bendIds, sc.bendId, st));
  PIES_CHECK(s, uploadVec(s->shapeOff, sc.shapeOff, st)); PIES_CHECK(s, uploadVec(s->shapeIds, sc.shapeId, st));
  PIES_CHECK(s, uploadVec(s->shapeMat, sc.shapeMat, st)); PIES_CHECK(s, uploadVec(s->shapeQinv, sc.shapeQinv, st));
  PIES_CHECK(s, uploadVec(s->shapeQuat, sc.shapeQuat, st)); PIES_CHECK(s, uploadVec(s->shapeW, sc.shapeW, st));
  PIES_CHECK(s, uploadVec(s->goalOff, sc.goalOff, st)); PIES_CHECK(s, uploadVec(s->goalIds, sc.goalId, st));
  PIES_CHECK(s, uploadVec(s->goalMat, sc.goalMat, st)); PIES_CHECK(s, uploadVec(s->goalW, sc.goalW, st));
  PIES_CHECK(s, s->goalXform.upload(reinterpret_cast<const float*>(sc.goalXform.data()), sc.goalXform.size() * 16, st));
  sc.goalXformDirty = false;
  PIES_CHECK(s, uploadVec(s->incPtr, y.incPtr, st)); PIES_CHECK(s, uploadVec(s->inc, y.inc, st));
  PIES_CHECK(s, uploadVec(s->segs, y.segs, st)); PIES_CHECK(s, uploadVec(s->segSlot, y.segSlot, st));
  PIES_CHECK(s, uploadVec(s->restElems, y.restElems, st)); PIES_CHECK(s, uploadVec(s->restNodes, y.restNodes, st));
  PIES_CHECK(s, uploadVec(s->rowPtr, y.rowPtr, st)); PIES_CHECK(s, uploadVec(s->col, y.col, st)); PIES_CHECK(s, uploadVec(s->val, y.val, st));
  PIES_CHECK(s, uploadVec(s->sellPtr, y.sellPtr, st)); PIES_CHECK(s, uploadVec(s->sellRow, y.sellRow, st));
  PIES_CHECK(s, uploadVec(s->sellCol, y.sellCol, st)); PIES_CHECK(s, uploadVec(s->sellVal, y.sellVal, st));
  PIES_CHECK(s, uploadVec(s->blockNodes, y.blockNodes, st)); PIES_CHECK(s, uploadVec(s->blockInv, y.blockInv, st));
  PIES_CHECK(s, uploadVec(s->triIds, sc.triangles, st));
  if (!s->islands) s->islands = new IslandWork();
  if (uploadIslandStatics(*s->islands, st, y) != 0) return failCuda(s, s->islands->lastError, "uploadIslandStatics", __LINE__);
  preloadDetectKernels(); preloadContactKernels(); preloadReblockKernels(); preloadSortKernels(); preloadPcgKernels();
  preloadIslandKernels(); preloadColliderKernels();
  {
    // The per-substep collision buffers (detect.cu, reblock.cu, contact.cu) first appear, and later grow, in the middle
    // of a run; growing the stream-ordered pool there costs tens of milliseconds in one tick.  Reserve the pool once
    // per topology instead: allocate and free a block sized for a contact-rich substep (the pool keeps freed memory,
    // capi.cpp sets its release threshold to "never").
    size_t freeB = 0, totalB = 0;
    if (cudaMemGetInfo(&freeB, &totalB) == cudaSuccess) {
      size_t want = std::max<size_t>(256ull << 20, 3072ull * sc.triCount() + 1024ull * n);
      want = std::min(want, freeB / 4);
      void* warm = nullptr;
      if (want && cudaMallocAsync(&warm, want, st) == cudaSuccess) cudaFreeAsync(warm, st);
    }
    cudaGetLastError();
  }
  PIES_CHECK(s, cudaStreamSynchronize(st));
  s->builtVersion = sc.topologyVersion;
  s->vtxDevValid = false;
  s->hostStateDirty = false;
  s->stats.staticProjections = y.staticProjections;
  s->stats.systemNonZeros = y.col.size();
  s->stats.staticBodies = y.nBodies;
  s->lastPcgIters = 1;
  return PIES_B200_OK;
}

// positions into the device copy of the Vertex mirror: 3 floats at the head of every 9-float record
__global__ void __launch_bounds__(kThreads) k_vertex_positions(uint32_t n, const float4* __restrict__ q, float* __restrict__ vtx) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 v = q[i];
  float* o = vtx + 9ull * i;
  o[0] = v.x; o[1] = v.y; o[2] = v.z;
}

void unregisterVertexMirror(PiesB200Solver* s) {
  if (s->vtxRegistered) { cudaHostUnregister(s->vtxRegistered); cudaGetLastError(); }
  s->vtxRegistered = nullptr; s->vtxRegisteredBytes = 0;
}

// Solver::getVertices (Solver.h:65): the reference refreshes _vertices[i].position on the host at the end of every substep
// (Solver.cpp:393); here the whole 36 B-stride mirror comes back in one DMA, no host-side scatter.
// Device-side Vertex array (internal, or the caller's render buffer): static attributes once per topology, positions now.
int refreshDeviceVertices(PiesB200Solver* s, float** out) {
  const uint32_t n = s->n;
  static_assert(sizeof(PiesB200Vertex) == 36, "Vertex is 9 floats");
  const size_t bytes = (size_t)n * sizeof(PiesB200Vertex);
  float* dev = s->vtxExternal;
  if (!dev) { PIES_CHECK(s, s->vtxDev.reserve(9ull * n)); dev = s->vtxDev.p; }
  if (!s->vtxDevValid) {  // colours, radii: static per topology
    PIES_CHECK(s, cudaMemcpyAsync(dev, s->scene.vertices.data(), bytes, cudaMemcpyHostToDevice, s->stream));
    s->vtxDevValid = true;
  }
  k_vertex_positions<<<gridFor(n, kThreads), kThreads, 0, s->stream>>>(n, s->q.p, dev);
  ++s->launches;
  *out = dev;
  return PIES_B200_OK;
}

int refreshVertexMirror(PiesB200Solver* s) {
  if (!s->n) return PIES_B200_OK;
  const uint32_t n = s->n;
  const size_t bytes = (size_t)n * sizeof(PiesB200Vertex);
  PiesB200Vertex* host = s->scene.vertices.data();
  float* dev = nullptr;
  int rc = refreshDeviceVertices(s, &dev);
  if (rc) return rc;
  if (s->vtxRegistered != host || s->vtxRegisteredBytes != bytes) {
    unregisterVertexMirror(s);
    if (cudaHostRegister(host, bytes, cudaHostRegisterDefault) == cudaSuccess) { s->vtxRegistered = host; s->vtxRegisteredBytes = bytes; }
    else cudaGetLastError();  // pageable destination: the runtime stages the copy, still no scatter
  }
  PIES_CHECK(s, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, s->stream));
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  s->mirrorStale = false;
  return PIES_B200_OK;
}

namespace {
// Phase timing with CUDA event pairs recorded on the solver stream and resolved after the
// tick's final synchronisation (no extra syncs inside the tick).  Enabled by tuning.reserved.
enum Phase { kPhOther = 0, kPhDetect, kPhLocal, kPhGlobal, kPhContact, kPhTetKernel, kPhSpmvKernel, kPhUpdateKernel, kPhGatherKernel, kPhIslandKernel, kPhHalo, kPhCount };
struct PhaseTimer {
  PiesB200Solver* s;
  bool on;
  std::vector<cudaEvent_t>& pool;
  std::vector<std::pair<int, size_t>> spans;  // (phase, index of the start event)
  size_t used = 0;
  explicit PhaseTimer(PiesB200Solver* s_, std::vector<cudaEvent_t>& pool_) : s(s_), on((s_->tune.reserved & 1u) != 0), pool(pool_) {}
  cudaEvent_t next() {
    if (used == pool.size()) { cudaEvent_t e; cudaEventCreate(&e); pool.push_back(e); }
    return pool[used++];
  }
  // spans may nest (a sampled kernel inside a phase): begin() returns the span to hand to end()
  int begin(int phase) {
    if (!on) return -1;
    spans.emplace_back(phase, used); cudaEventRecord(next(), s->stream); next();
    return (int)spans.size() - 1;
  }
  void end(int span = -1) {
    if (!on) return;
    const auto& sp = span >= 0 ? spans[span] : spans.back();
    cudaEventRecord(pool[sp.second + 1], s->stream);
  }
  void discard(int span) { if (on && span >= 0) spans[span].first = -1; }  // e.g. a sampled launch that turned out to be an early exit
  void resolve(float (&acc)[kPhCount], uint32_t (&cnt)[kPhCount]) {
    for (auto& sp : spans) {
      if (sp.first < 0) continue;
      float ms = 0.0f;
      if (cudaEventElapsedTime(&ms, pool[sp.second], pool[sp.second + 1]) == cudaSuccess) { acc[sp.first] += ms; ++cnt[sp.first]; }
    }
  }
};
}  // namespace

int runDetection(PiesB200Solver* s, ContactLists& lists) {
  if (!s->detect) {
    s->detect = new DetectWork();
    PIES_CHECK(s, cudaMallocHost(&s->detect->host, 16 * sizeof(int)));
  }
  if (!s->contact) s->contact = new ContactWork();
  DetectInput in{s->triIds.p, s->q.p, s->prev.p, s->scene.triCount(), s->n, s->opt.threadCount,
                 s->opt.collisionThresholdDistance, s->opt.floorHeight + s->opt.collisionThickness,
                 (s->haveTriOrder && s->triOrder.cap >= s->scene.triCount()) ? s->triOrder.p : nullptr};
  in.colliders = colliderSet(s);
  in.thickness = s->opt.collisionThickness;
  if (in.colliders.n) {
    PIES_CHECK(s, s->colMask.reserve(s->n + 1)); PIES_CHECK(s, s->colRhs.reserve(s->n + 1));
    in.colMask = s->colMask.p;
  }
  in.drags = dragSet(s);
  in.msn = s->msn.p;
  int L = 0;
  lists = ContactLists{};
  if (detectTriangles(*s->detect, s->stream, in, lists, &L) != 0)
    return failCuda(s, s->detect->lastError, "detectTriangles", __LINE__);
  s->launches += L;
  PIES_CHECK(s, cudaGetLastError());
  if (s->detect->badInput) { s->simFailed = true; return fail(s, PIES_B200_ERANGE, "non-finite or out-of-range (|x| >= 2^30) positions reached collision detection"); }
  if (s->detect->failed) { s->simFailed = true; lists.nTri = lists.nFloor = 0; }  // Solver.cpp:852-856
  if (prepareContactSweeps(*s->contact, s->stream, lists) < 0)
    return failCuda(s, cudaErrorMemoryAllocation, "prepareContactSweeps", __LINE__);
  if (lists.nUnique) PIES_CHECK(s, s->contact->contribC.reserve(4ull * lists.nUnique));
  lists.colRhs = lists.nCollide ? s->colRhs.p : nullptr;
  s->colMaskColliders = lists.nCollide;
  s->stats.triCollisions = lists.nTri;
  s->stats.staticCollisions = lists.nFloor;
  return PIES_B200_OK;
}

// ---- PD tick, split into phases so a slab-partitioned host can exchange halos between them (DESIGN.md section 7).
// tickPD() below is the plain composition; the C ABI also exposes the phases (pies_b200_pd_*).
struct PdTickCtx {
  PhaseTimer timer;
  cudaEvent_t tick0 = nullptr, tick1 = nullptr;
  uint64_t launches0 = 0;
  ContactLists lists;
  bool inSubstep = false;
  uint32_t iterIndex = 0;  // PD iteration inside the current substep
  uint32_t solveIndex = 0; // global solves so far in this tick (record of IslandWork::solveStats)
  uint64_t globalIters = 0;  // per solve: CG iterations of the grid-wide solve, kept to combine with the island counts
  std::vector<uint32_t> globalItersPerSolve;
  PdTickCtx(PiesB200Solver* s) : timer(s, s->eventPool) {}
};

void pdAbort(PiesB200Solver* s) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  if (!c) return;
  delete c;  // the tick events belong to the solver
  s->pdCtx = nullptr;
}

namespace {
struct PdViews {
  TetElems te; DistanceElems de; BendElems be; ClusterElems sh, go; CsrMatrix A; PcgWork pw;
};
PdViews pdViews(PiesB200Solver* s) {
  const HostSystem& y = s->sys;
  PdViews v;
  v.te = TetElems{s->elemIds.p, s->elemQa.p, s->elemQb.p, s->elemPc.p, s->elemPd.p, (s->tune.reserved & 512u) ? nullptr : s->elemRot.p, y.nElems};
  v.de = DistanceElems{s->distIds.p, s->distRestW.p, (uint32_t)s->scene.distW.size()};
  v.be = BendElems{s->bendIds.p, s->bendAngleW.p, (uint32_t)s->scene.bendW.size()};
  v.sh = ClusterElems{s->shapeOff.p, s->shapeIds.p, (uint32_t)s->scene.shapeW.size(), (uint32_t)s->scene.shapeId.size()};
  v.go = ClusterElems{s->goalOff.p, s->goalIds.p, (uint32_t)s->scene.goalW.size(), (uint32_t)s->scene.goalId.size()};
  v.A = CsrMatrix{s->rowPtr.p, s->col.p, s->val.p, s->n, (uint64_t)y.col.size(), s->sellPtr.p, s->sellRow.p, s->sellCol.p,
                  s->sellVal.p, (uint32_t)(y.sellPtr.empty() ? 0 : y.sellPtr.size() - 1), (uint64_t)y.sellVal.size()};
  v.pw.r = s->pr.p; v.pw.p = s->pp.p; v.pw.p2 = s->pp2.p; v.pw.z = s->pz.p; v.pw.ap = s->pap.p; v.pw.delta = s->pdelta.p;
  v.pw.partials = s->partials.p; v.pw.scalars = s->scalars.p; v.pw.flag = s->flag.p;
  if (s->blocks) {  // the contact-aware blocks of the current substep (reblock.cu)
    v.pw.blockNodes = s->blocks->cur.blockNodes; v.pw.blockInv = s->blocks->cur.blockInv;
    v.pw.blockMeta = s->blocks->cur.blockMeta; v.pw.nBlocks = s->blocks->cur.nBlocks; v.pw.nBlocksDev = s->blocks->cur.nBlocksDev;
  }
  return v;
}
}  // namespace

int pdTickBegin(PiesB200Solver* s) {
  pdAbort(s);
  int rc = ensureBuilt(s);
  if (rc) return rc;
  s->stats.substepsLastTick = 0;
  s->stats.projectionsLastTick = 0;
  s->stats.pcgIterationsLastTick = 0;
  s->stats.msLocal = s->stats.msGlobal = s->stats.msDetect = s->stats.msContact = s->stats.msOther = 0.0f;
  s->stats.msTetKernel = 0.0f; s->stats.tetKernelLaunches = 0;
  s->stats.msSpmvKernel = s->stats.msUpdateKernel = s->stats.msGatherKernel = 0.0f;
  s->stats.spmvKernelLaunches = s->stats.updateKernelLaunches = s->stats.gatherKernelLaunches = 0;
  s->stats.pcgCapHits = 0; s->stats.pcgWorstCapResidual = 0.0f; s->stats.msIslandKernels = 0.0f;
  s->stats.islandKernelLaunches = 0; s->stats.pcgIslandRowIterations = 0;
  s->stats.msHalo = 0.0f; s->stats.haloBytesLastTick = 0; s->stats.haloExchangesLastTick = 0;
  PdTickCtx* c = new PdTickCtx(s);
  c->launches0 = s->launches;
  s->pdCtx = c;
  if (!s->n) return PIES_B200_OK;
  if ((rc = prepareForces(s))) { pdAbort(s); return rc; }
  if (s->islands) {
    const size_t words = 4ull * s->opt.timeSubsteps * s->opt.iterations + 4;
    PIES_CHECK(s, s->islands->solveStats.reserve(words));
    PIES_CHECK(s, cudaMemsetAsync(s->islands->solveStats.p, 0, words * sizeof(uint32_t), s->stream));
  }
  if ((rc = ensureTickEvents(s))) { pdAbort(s); return rc; }
  c->tick0 = s->tickEv[0]; c->tick1 = s->tickEv[1];
  cudaEventRecord(c->tick0, s->stream);
  return PIES_B200_OK;
}

// PIES_CHECK inside a tick phase: drops the tick context before returning the error
#define PD_CHECK(s, expr)                                                          \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) { pdAbort(s); return failCuda((s), _e, #expr, __LINE__); } \
  } while (0)

int pdSubstepBegin(PiesB200Solver* s) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  if (!c) return fail(s, PIES_B200_EINVAL, "pd_substep_begin outside pd_tick_begin/pd_tick_end");
  const uint32_t n = s->n;
  if (!n) { c->inSubstep = true; return PIES_B200_OK; }  // empty scene: the phases are no-ops but stay well-formed
  cudaStream_t st = s->stream;
  const PiesB200Options& o = s->opt;
  const float h = o.fixedTimestepSize / (float)o.timeSubsteps;
  PhaseTimer& timer = c->timer;
  int rc;
  timer.begin(kPhOther);
  s->launches += launchForces(st, n, forceSet(s), s->q.p, s->vel.p);   // on the substep-start q and vel
  s->launches += launchPredict(st, n, s->q.p, s->vel.p, s->msn.p, h);
  timer.end();

  timer.begin(kPhDetect);
  if ((rc = runDetection(s, c->lists))) { pdAbort(s); return rc; }
  // contact-aware preconditioner blocks for this substep's system matrix S + C_t
  if (!s->blocks) {
    s->blocks = new BlockWork();
    PD_CHECK(s, cudaMallocHost(&s->blocks->host, 4 * sizeof(uint32_t)));
  }
  s->blocks->midClusterMax = (s->tune.reserved & 2u) ? 0u : kMidClusterMax;
  {
    PdViews v = pdViews(s);
    int LB = 0;
    if (rebuildBlocks(*s->blocks, st, n, v.A, s->blockNodes.p, s->blockInv.p, s->sys.nBlocks, c->lists, s->q.p, v.pw, &LB) != 0) {
      cudaError_t e = s->blocks->lastError;
      pdAbort(s);
      return failCuda(s, e, "rebuildBlocks", __LINE__);
    }
    s->blocks->cur.blockNodes = v.pw.blockNodes; s->blocks->cur.blockInv = v.pw.blockInv; s->blocks->cur.blockMeta = v.pw.blockMeta;
    s->blocks->cur.nBlocks = v.pw.nBlocks; s->blocks->cur.nBlocksDev = v.pw.nBlocksDev;
    s->launches += LB;
    const BlockWork& bw = *s->blocks;
    ClusterTables ct{bw.heads.p + bw.nTouched, bw.start.p, bw.vals.p, bw.clusterOf.p, bw.rankOf.p, bw.gsClass.p, bw.nTouched,
                     bw.midList.p, bw.midCount.p, bw.host + 1, bw.countsReady};
    int LC = s->contact ? prepareClusterSweeps(*s->contact, st, c->lists, ct) : 0;
    if (LC < 0) { pdAbort(s); return failCuda(s, cudaErrorMemoryAllocation, "prepareClusterSweeps", __LINE__); }
    s->launches += LC;
    // islands of S + C_t: which solves stay inside one warp / one CTA (islands.cu)
    if (s->islands) {
      int LI = 0;
      if (buildIslands(*s->islands, st, n, v.A, c->lists, bw.slotOf.p, bw.blockCount.p, bw.nBlocksBound, s->tune.reserved, &LI) != 0) {
        cudaError_t e = s->islands->lastError;
        pdAbort(s);
        return failCuda(s, e, "buildIslands", __LINE__);
      }
      s->launches += LI;
      islandStats(*s->islands, s->stats);
    }
  }
  timer.end();
  c->inSubstep = true;
  c->iterIndex = 0;
  return PIES_B200_OK;
}

int pdIteration(PiesB200Solver* s) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  if (!c || !c->inSubstep) return fail(s, PIES_B200_EINVAL, "pd_iteration outside a substep");
  const uint32_t n = s->n;
  if (!n) return PIES_B200_OK;
  cudaStream_t st = s->stream;
  const HostSystem& y = s->sys;
  PhaseTimer& timer = c->timer;
  const ContactLists& lists = c->lists;
  PdViews v = pdViews(s);
  float4* contribC = s->contact ? s->contact->contribC.p : nullptr;
  const bool anyContact = lists.nTri || lists.nodeWeights();
  // The fused local step + RHS (k_tet_rhs) covers the closed segments; the elements and nodes outside them take the
  // two-kernel path.  A/B switch: PIES_B200_NO_FUSED_LOCAL sends everything through the two-kernel path.
  static const bool noFused = std::getenv("PIES_B200_NO_FUSED_LOCAL") != nullptr;
  const bool fused = !noFused && !y.segs.empty();
  const TetSegments sg{s->segs.p, s->segSlot.p, fused ? (uint32_t)(y.segs.size() / 4) : 0u};
  const uint32_t* tetList = fused ? s->restElems.p : nullptr;
  const uint32_t* nodeList = fused ? s->restNodes.p : nullptr;
  const uint32_t nTetList = fused ? (uint32_t)y.restElems.size() : y.nElems;
  const uint32_t nNodeList = fused ? (uint32_t)y.restNodes.size() : n;
  // the local span holds the tet span (msLocal is the whole local step + RHS)
  const int spLocal = timer.begin(kPhLocal);
  s->launches += launchContactProject(st, lists, s->q.p, s->opt.collisionThickness, contribC);  // k_tet_rhs reads contribC
  if (lists.nCollide)   // ... and colRhs
    s->launches += launchColliderProject(st, n, colliderSet(s), lists.colMask, s->q.p, s->colRhs.p);
  // the tet slot times the tet projections of both paths, with the RHS of the segments when fused
  const int spTet = timer.begin(kPhTetKernel);
  s->launches += launchTetRhs(st, v.te, sg, s->q.p, s->msn.p, s->incPtr.p, lists, contribC, s->snap.p, s->rhs.p);
  s->launches += launchTetElems(st, v.te, tetList, nTetList, s->q.p, s->contrib.p + y.baseTet);
  timer.end(spTet);
  s->launches += launchDistance(st, v.de, s->q.p, s->contrib.p + y.baseDist);
  s->launches += launchBend(st, v.be, s->q.p, s->contrib.p + y.baseBend);
  s->launches += launchShape(st, v.sh, s->shapeMat.p, s->shapeQinv.p, s->shapeQuat.p, s->shapeW.p, s->q.p, s->contrib.p + y.baseShape);
  s->launches += launchGoal(st, v.go, s->goalMat.p, s->goalXform.p, s->goalW.p, s->contrib.p + y.baseGoal);
  if (nNodeList) {
    const int spGather = timer.begin(kPhGatherKernel);
    if (anyContact)   // constraints + collision + floor terms in one pass over the nodes (it also writes the floor snap)
      s->launches += launchGatherRhsContacts(st, nNodeList, nodeList, s->msn.p, s->incPtr.p, s->inc.p, s->contrib.p, lists,
                                             contribC, s->q.p, s->snap.p, s->rhs.p);
    else
      s->launches += launchGatherRhs(st, nNodeList, nodeList, s->msn.p, s->incPtr.p, s->inc.p, s->contrib.p, s->rhs.p);
    timer.end(spGather);
  }
  timer.end(spLocal);

  const int spGlobal = timer.begin(kPhGlobal);
  if (s->blocks && s->blocks->factorPending) {   // this substep's block inverses (side stream of rebuildBlocks)
    PD_CHECK(s, cudaStreamWaitEvent(st, s->blocks->factorDone, 0));
    s->blocks->factorPending = false;
  }
  const uint32_t k = c->iterIndex++;
  const uint32_t solveSlot = c->solveIndex++;
  uint32_t used = 0;
  bool gridWide = true;
  if (s->islands && s->blocks) {
    IslandWork& iw = *s->islands;
    if (iw.anyLocal()) {
      const int spIsl = timer.begin(kPhIslandKernel);
      s->launches += launchIslandSolve(iw, st, v.A, lists, v.pw, s->blocks->slotOf.p, s->rhs.p, s->q.p, s->tune.pcgTolerance,
                                       s->tune.pcgMaxIterations, solveSlot);
      timer.end(spIsl);
    }
    gridWide = iw.nLeftIslands != 0;
    if (gridWide) applyRestriction(iw, v.pw);  // only the rows of the left-over islands
  }
  if (gridWide) {
    int spSpmv = -1, spUpdate = -1;  // one sampled CG iteration (the second of the solve) per PD iteration
    s->launches += launchPcgInit(st, v.A, lists, v.pw, s->rhs.p, s->q.p, s->tune.pcgTolerance);
    // Iterations are enqueued in bursts without host round trips: converged solves turn the remaining
    // launches into early exits (~2 us each), a host poll costs ~40 us of idle GPU, so the first burst
    // slightly overshoots the previous solve's count.
    // The k-th PD iteration of a substep needs about what the k-th of the previous substep needed (the first solve after
    // the inertia step more than the later ones), which predicts the burst better than the previous solve of this substep.
    if (s->pcgItersByIteration.size() <= k) s->pcgItersByIteration.resize(k + 1, s->lastPcgIters);
    uint32_t done = 0, burst = s->pcgItersByIteration[k] + 1;
    bool converged = false;
    while (!converged && done < s->tune.pcgMaxIterations) {
      uint32_t todo = std::min(burst, s->tune.pcgMaxIterations - done);
      for (uint32_t j = 0; j < todo; ++j) {
        const int it = (int)(done + j);
        if (it == 1 && timer.on) {
          spSpmv = timer.begin(kPhSpmvKernel);
          s->launches += launchPcgSpmv(st, v.A, lists, v.pw, s->tune.pcgTolerance, it);
          timer.end(spSpmv);
          spUpdate = timer.begin(kPhUpdateKernel);
          s->launches += launchPcgUpdate(st, v.pw, s->tune.pcgTolerance, it);
          timer.end(spUpdate);
        } else {
          s->launches += launchPcgIteration(st, v.A, lists, v.pw, s->tune.pcgTolerance, it);
        }
      }
      done += todo;
      s->launches += launchPcgCheck(st, v.pw, s->tune.pcgTolerance, (int)done - 1);
      PD_CHECK(s, cudaMemcpyAsync(s->hostFlag, s->flag.p, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
      PD_CHECK(s, cudaMemcpyAsync(s->hostFlag + 2, s->scalars.p, sizeof(float), cudaMemcpyDeviceToHost, st));
      PD_CHECK(s, cudaStreamSynchronize(st));
      converged = s->hostFlag[0] != 0;
      burst = std::max(4u, s->tune.pcgCheckEvery);
    }
    s->launches += launchPcgFinish(st, v.pw, n, s->q.p);
    used = (uint32_t)s->hostFlag[1];
    if (getenv("PIES_DEBUG_PCG")) std::fprintf(stderr, "[pcg] it: %u iterations\n", used);
    s->lastPcgIters = std::max(1u, used);
    s->pcgItersByIteration[k] = s->lastPcgIters;
    if (used < 2) { timer.discard(spSpmv); timer.discard(spUpdate); }  // the sampled launches were early exits
    float rel;
    std::memcpy(&rel, s->hostFlag + 2, sizeof(float));
    s->stats.pcgLastRelResidual = rel;
    if (!converged) {  // stopped at the cap: say so (pdTickEnd turns a residual far above the tolerance into an error)
      ++s->stats.pcgCapHits;
      s->stats.pcgWorstCapResidual = std::max(s->stats.pcgWorstCapResidual, rel);
    }
  }
  c->globalItersPerSolve.push_back(used);
  timer.end(spGlobal);
  s->stats.projectionsLastTick += y.staticProjections + lists.nTri + lists.nFloor;
  return PIES_B200_OK;
}

int pdSubstepEnd(PiesB200Solver* s) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  if (!c || !c->inSubstep) return fail(s, PIES_B200_EINVAL, "pd_substep_end outside a substep");
  c->inSubstep = false;
  const uint32_t n = s->n;
  if (!n) return PIES_B200_OK;
  cudaStream_t st = s->stream;
  const PiesB200Options& o = s->opt;
  const float h = o.fixedTimestepSize / (float)o.timeSubsteps;
  PhaseTimer& timer = c->timer;
  const ContactLists& lists = c->lists;
  // nothing of this substep's side-stream preparation may outlive it (a substep without PD iterations never waited)
  if (s->blocks && s->blocks->factorPending) { PD_CHECK(s, cudaStreamWaitEvent(st, s->blocks->factorDone, 0)); s->blocks->factorPending = false; }
  timer.begin(kPhContact);
  if (s->contact)
    s->launches += launchStabilize(st, *s->contact, lists, n, s->q.p, s->prev.p, s->snap.p, o.collisionThickness,
                                   o.collisionStabilizationIterations);
  if (lists.nCollide) s->launches += launchColliderSnap(st, n, colliderSet(s), lists.colMask, s->q.p);
  timer.end();
  s->stats.reserved = 0;
  if (s->blocks && s->blocks->countsReady && lists.nTri) {
    cudaEventSynchronize(s->blocks->countsReady);
    s->stats.reserved = std::min(s->blocks->host[1], 65535u) | (std::min(s->blocks->host[2], 65535u) << 16);
  }
  timer.begin(kPhOther);
  s->launches += launchVelocityUpdate(st, n, s->q.p, s->prev.p, s->vel.p, h, o.damping, o.gravity, forceSet(s).field());
  timer.end();
  timer.begin(kPhContact);
  if (s->contact) s->launches += launchFriction(st, *s->contact, lists, n, s->q.p, s->vel.p, o.friction, o.staticFrictionThreshold);
  if (lists.nCollide)
    s->launches += launchColliderFriction(st, n, colliderSet(s), lists.colMask, s->q.p, s->vel.p, o.friction, o.staticFrictionThreshold);
  timer.end();
  s->stats.collisionProjections = lists.nTri + lists.nFloor;
  ++s->stats.substepsLastTick;
  return PIES_B200_OK;
}

int pdTickEnd(PiesB200Solver* s, bool refreshMirror) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  if (!c) return fail(s, PIES_B200_EINVAL, "pd_tick_end without pd_tick_begin");
  if (!s->n) { pdAbort(s); return PIES_B200_OK; }
  cudaStream_t st = s->stream;
  s->deviceNewer = true;
  cudaEventRecord(c->tick1, st);
  cudaError_t es = cudaEventSynchronize(c->tick1);
  if (es != cudaSuccess) { pdAbort(s); return failCuda(s, es, "cudaEventSynchronize", __LINE__); }
  cudaEventElapsedTime(&s->stats.msTick, c->tick0, c->tick1);
  {
    float acc[kPhCount] = {};
    uint32_t cnt[kPhCount] = {};
    c->timer.resolve(acc, cnt);
    s->stats.msOther = acc[kPhOther]; s->stats.msDetect = acc[kPhDetect]; s->stats.msLocal = acc[kPhLocal];
    s->stats.msGlobal = acc[kPhGlobal]; s->stats.msContact = acc[kPhContact];
    s->stats.msTetKernel = acc[kPhTetKernel]; s->stats.tetKernelLaunches = cnt[kPhTetKernel];
    s->stats.msSpmvKernel = acc[kPhSpmvKernel]; s->stats.spmvKernelLaunches = cnt[kPhSpmvKernel];
    s->stats.msUpdateKernel = acc[kPhUpdateKernel]; s->stats.updateKernelLaunches = cnt[kPhUpdateKernel];
    s->stats.msGatherKernel = acc[kPhGatherKernel]; s->stats.gatherKernelLaunches = cnt[kPhGatherKernel];
    s->stats.msIslandKernels = acc[kPhIslandKernel]; s->stats.islandKernelLaunches = cnt[kPhIslandKernel];
    s->stats.msHalo = acc[kPhHalo];
  }
  uint64_t launches0 = c->launches0;
  const std::vector<uint32_t> solves = c->globalItersPerSolve;
  pdAbort(s);
  PIES_CHECK(s, cudaGetLastError());
  int rcConv = PIES_B200_OK;
  {
    // per-solve records of the island kernels (max iterations, work, islands stopped at the cap, their worst residual)
    // combined with the grid-wide CG's counts: a solve took as many iterations as its slowest part
    const size_t nSolves = solves.size();
    std::vector<uint32_t> rec(4 * nSolves + 4, 0u);
    if (s->islands && s->islands->solveStats.p && nSolves)
      PIES_CHECK(s, cudaMemcpy(rec.data(), s->islands->solveStats.p, 4 * nSolves * sizeof(uint32_t), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < nSolves; ++i) {
      s->stats.pcgIterationsLastTick += std::max(solves[i], rec[4 * i]);
      s->stats.pcgIslandRowIterations += rec[4 * i + 1];
      if (rec[4 * i + 2]) {
        s->stats.pcgCapHits += rec[4 * i + 2];
        float rel;
        std::memcpy(&rel, &rec[4 * i + 3], sizeof(float));
        s->stats.pcgWorstCapResidual = std::max(s->stats.pcgWorstCapResidual, rel);
      }
    }
    // Stopping at the cap a little above the tolerance is fp32 stagnation and only counted; far above it the solve
    // did not converge and the caller must know (the reference's Cholesky cannot fail this way).
    if (s->stats.pcgCapHits && s->stats.pcgWorstCapResidual > 1000.0f * s->tune.pcgTolerance) {
      char buf[256];
      std::snprintf(buf, sizeof(buf), "global solve not converged: %u solves stopped at pcgMaxIterations = %u, worst relative residual %.3g (tolerance %.3g)",
                    s->stats.pcgCapHits, s->tune.pcgMaxIterations, s->stats.pcgWorstCapResidual, s->tune.pcgTolerance);
      s->err = buf;
      rcConv = PIES_B200_ENOCONV;
    }
  }
  s->mirrorStale = true;
  int rc;
  if (refreshMirror && (rc = refreshVertexMirror(s))) return rc;
  s->stats.kernelLaunchesLastTick = s->launches - launches0;
  s->stats.simFailed = s->simFailed ? 1u : 0u;
  return rcConv;
}

// contacts of the last detection whose point node (point-triangle) / node (floor) this solver owns
__global__ void __launch_bounds__(kThreads) k_count_owned(uint32_t nTri, const uint4* __restrict__ tri, uint32_t nFloor,
                                                          const uint32_t* __restrict__ floorNode,
                                                          const uint8_t* __restrict__ owned, uint32_t* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t a = 0, b = 0;
  if (i < nTri) a = owned[tri[i].x] ? 1u : 0u;
  if (i < nFloor) b = owned[floorNode[i]] ? 1u : 0u;
  a = __reduce_add_sync(0xffffffffu, a); b = __reduce_add_sync(0xffffffffu, b);
  if ((threadIdx.x & 31) == 0) { if (a) atomicAdd(out, a); if (b) atomicAdd(out + 1, b); }
}

int countOwnedContacts(PiesB200Solver* s, uint32_t* nTri, uint32_t* nFloor) {
  *nTri = s->stats.triCollisions; *nFloor = s->stats.staticCollisions;
  if (!s->haveOwnedMask || !s->detect || (!*nTri && !*nFloor)) return PIES_B200_OK;
  uint32_t m = std::max(*nTri, *nFloor);
  // NOT s->flag: flag[2] is the ticket counter of the CG kernels' grid reductions and must stay 0 between kernels
  PIES_CHECK(s, s->ownedCount.reserve(2));
  uint32_t* out = s->ownedCount.p;
  PIES_CHECK(s, cudaMemsetAsync(out, 0, 2 * sizeof(uint32_t), s->stream));
  k_count_owned<<<gridFor(m, kThreads), kThreads, 0, s->stream>>>(*nTri, s->detect->triList.p, *nFloor, s->detect->floorList.p,
                                                                 s->ownedMask.p, out);
  ++s->launches;
  uint32_t host[2] = {0, 0};
  PIES_CHECK(s, cudaMemcpyAsync(host, out, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  *nTri = host[0]; *nFloor = host[1];
  return PIES_B200_OK;
}

// One halo exchange inside a tick (slab-partitioned runs), timed as its own phase.
static int tickHalo(PiesB200Solver* s, int planes) {
  PdTickCtx* c = static_cast<PdTickCtx*>(s->pdCtx);
  int span = c ? c->timer.begin(kPhHalo) : -1;
  int rc = haloExchange(s, planes);
  if (c) c->timer.end(span);
  return rc;
}

int tickPD(PiesB200Solver* s, bool refreshMirror) {
  const bool multi = s->halo && s->halo->world > 1;
  if (multi) {
    // every rank takes part in this reduction at every tick, failed or not, so that they all stop at the same tick:
    // a rank that went on alone would wait for its neighbours' halos forever
    bool any = false;
    int rcf = haloAnyFailed(s, s->simFailed, &any);
    if (rcf) return rcf;
    if (any) { s->simFailed = true; s->stats.simFailed = 1u; return PIES_B200_OK; }  // Solver.cpp:26-28: silent no-op once failed
    s->halo->bytesLastTick = 0; s->halo->exchangesLastTick = 0;
  }
  int rc = pdTickBegin(s);
  if (rc) return rc;
  // After a failure in the middle of a tick a slab rank keeps its place in the communication pattern (its neighbours are
  // waiting in the matching exchanges) and only skips the compute; the next tick's reduction stops every rank.
  int failed = PIES_B200_OK;
  for (uint32_t sub = 0; sub < s->opt.timeSubsteps; ++sub) {
    if (multi && (rc = tickHalo(s, 3))) return rc;
    if (!failed && (rc = pdSubstepBegin(s))) { pdAbort(s); failed = rc; if (!multi) return rc; }
    // No island mixes owned and ghost rows on any rank (agreed collectively): the owned rows do not see the ghost rows
    // for the rest of the substep, so the exchange after every PD iteration is skipped.
    bool mixed = true;
    if (multi && (rc = haloMixedIslands(s, !failed, &mixed))) return rc;
    for (uint32_t it = 0; it < s->opt.iterations; ++it) {
      if (!failed && (rc = pdIteration(s))) { pdAbort(s); failed = rc; if (!multi) return rc; }
      if (multi && mixed && (rc = tickHalo(s, 1))) return rc;
    }
    if (!failed && (rc = pdSubstepEnd(s))) { pdAbort(s); failed = rc; if (!multi) return rc; }
  }
  if (failed) { s->simFailed = true; return failed; }
  rc = pdTickEnd(s, refreshMirror);
  if (multi) { s->stats.haloBytesLastTick = s->halo->bytesLastTick; s->stats.haloExchangesLastTick = (uint32_t)s->halo->exchangesLastTick; }
  return rc;
}

}  // namespace pies

PiesB200Solver::~PiesB200Solver() {
  if (detect) { if (detect->host) cudaFreeHost(detect->host); delete detect; }
  delete contact;
  pies::destroyPbdWork(pbd);
  pies::pdAbort(this);
  if (blocks) { if (blocks->host) cudaFreeHost(blocks->host); delete blocks; }
  delete islands;
  delete halo;
  pies::unregisterVertexMirror(this);
  for (cudaEvent_t e : eventPool) cudaEventDestroy(e);
  for (cudaEvent_t e : tickEv) if (e) cudaEventDestroy(e);
  if (hostPacked) cudaFreeHost(hostPacked);
  if (hostFlag) cudaFreeHost(hostFlag);
  if (ownStream && stream) cudaStreamDestroy(stream);
}
