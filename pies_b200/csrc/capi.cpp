// capi.cpp — the extern "C" boundary declared in include/pies_b200.h.
// Thin: argument checks, host-state synchronisation before scene mutations, and
// forwarding to the engine.  Never throws across the boundary.
#include <cstring>
#include <new>
#include <string>

#include "contact.h"
#include "detect.h"
#include <cstdlib>

#include "engine.h"
#include "halo.h"
#include "islands.h"

using pies::fail;

static std::string g_createError;

namespace {
template <typename F>
int guarded(PiesB200Solver* s, F&& f) {
  if (!s) return PIES_B200_EINVAL;
  try {
    cudaSetDevice(s->device);
    pies::g_allocStream = s->stream;  // device buffers grow on the caller's stream (engine.h: DevBuf)
    return f();
  } catch (const std::bad_alloc&) {
    return fail(s, PIES_B200_ERANGE, "host allocation failed");
  } catch (const std::exception& e) {
    return fail(s, PIES_B200_EINVAL, e.what());
  } catch (...) {
    return fail(s, PIES_B200_EINVAL, "unknown exception");
  }
}
// Scene mutations read current node positions (rest lengths, Qinv, region membership), so the
// host copy has to be brought up to date with the device first.
template <typename F>
int mutate(PiesB200Solver* s, F&& f) {
  return guarded(s, [&]() {
    int rc = pies::downloadState(s);
    if (rc) return rc;
    pies::unregisterVertexMirror(s);  // the factories grow scene.vertices
    f();
    s->renderStateDirty = true;
    return PIES_B200_OK;
  });
}
bool validIds(const PiesB200Solver* s, const uint32_t* ids, size_t count) {
  uint32_t n = s->scene.nodeCount();
  for (size_t i = 0; i < count; ++i) if (ids[i] >= n) return false;
  return true;
}
}  // namespace

extern "C" {

void pies_b200_default_options(PiesB200Options* o) {
  if (!o) return;
  o->fixedTimestepSize = 0.012f; o->timeSubsteps = 1; o->iterations = 4; o->collisionStabilizationIterations = 4;
  o->collisionThresholdDistance = 0.1f; o->collisionThickness = 0.05f; o->gravity = 10.0f; o->damping = 0.006f;
  o->friction = 0.01f; o->staticFrictionThreshold = 0.0f; o->floorHeight = 0.0f; o->gridSpacing = 2.0f;
  o->threadCount = 8; o->solver = 1;
}

void pies_b200_default_tuning(PiesB200Tuning* t) {
  if (!t) return;
  t->pcgTolerance = 1e-7f; t->pcgMaxIterations = 200; t->pcgCheckEvery = 1; t->reserved = 0;
  // experiment hook: PIES_B200_PCG_TOL overrides the default stopping tolerance (hosts use pies_b200_set_tuning)
  if (const char* e = std::getenv("PIES_B200_PCG_TOL")) { float v = (float)std::atof(e); if (v > 0.0f && v < 1.0f) t->pcgTolerance = v; }
}

int pies_b200_create(const PiesB200Options* options, int device, PiesB200Solver** out) {
  if (!out) return PIES_B200_EINVAL;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_createError = std::string("no CUDA device (") + cudaGetErrorString(e) + "); pies_b200 has no CPU fallback";
    cudaGetLastError();
    return PIES_B200_ENODEV;
  }
  if (device < 0) cudaGetDevice(&device);
  if (device >= count) { g_createError = "device index out of range"; return PIES_B200_EINVAL; }
  cudaDeviceProp prop{};
  cudaGetDeviceProperties(&prop, device);
  if (prop.major < 10) {
    g_createError = std::string("device '") + prop.name + "' is not sm_100; the kernels are built for sm_100a only";
    return PIES_B200_ENODEV;
  }
  PiesB200Solver* s = new (std::nothrow) PiesB200Solver();
  if (!s) { g_createError = "out of host memory"; return PIES_B200_ERANGE; }
  if (options) s->opt = *options; else pies_b200_default_options(&s->opt);
  if (s->opt.timeSubsteps == 0) s->opt.timeSubsteps = 1;
  pies_b200_default_tuning(&s->tune);
  s->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMallocHost(&s->hostFlag, 4 * sizeof(int)) != cudaSuccess) {
    g_createError = std::string("CUDA initialisation failed: ") + cudaGetErrorString(cudaGetLastError());
    delete s;
    return PIES_B200_ECUDA;
  }
  s->ownStream = true;
  s->hostFlag[0] = s->hostFlag[1] = 0;
  {  // keep freed device blocks cached in the default pool instead of returning them to the driver at every sync
    cudaMemPool_t pool = nullptr;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess && pool) {
      unsigned long long keep = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
    }
    cudaGetLastError();
  }
  *out = s;
  return PIES_B200_OK;
}

void pies_b200_destroy(PiesB200Solver* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  cudaStreamSynchronize(s->stream);
  delete s;
}

const char* pies_b200_last_error(const PiesB200Solver* s) { return s ? s->err.c_str() : g_createError.c_str(); }

int pies_b200_set_tuning(PiesB200Solver* s, const PiesB200Tuning* t) {
  if (!s || !t) return PIES_B200_EINVAL;
  s->tune = *t;
  if (s->tune.pcgMaxIterations == 0) s->tune.pcgMaxIterations = 1;
  if (s->tune.pcgCheckEvery == 0) s->tune.pcgCheckEvery = 1;
  return PIES_B200_OK;
}

int pies_b200_set_stream(PiesB200Solver* s, void* stream) {
  if (!s) return PIES_B200_EINVAL;
  cudaStreamSynchronize(s->stream);
  if (s->ownStream && s->stream) cudaStreamDestroy(s->stream);
  s->stream = reinterpret_cast<cudaStream_t>(stream);
  s->ownStream = false;
  return PIES_B200_OK;
}

int pies_b200_get_options(const PiesB200Solver* s, PiesB200Options* out) {
  if (!s || !out) return PIES_B200_EINVAL;
  *out = s->opt;
  return PIES_B200_OK;
}

// ---- stepping ----
static int tickOnce(PiesB200Solver* s, int which, bool refresh) {
  // Solver.cpp:26-28: silent no-op once failed (a slab rank still joins its peers' failure reduction inside tickPD)
  if (s->simFailed && !(which != 0 && s->halo && s->halo->world > 1)) return PIES_B200_OK;
  cudaSetDevice(s->device);
  (void)refresh;  // the vertex mirror is refreshed lazily by pies_b200_get_vertices
  if (which == 0) return pies::tickPBD(s, false);
  return pies::tickPD(s, false);
}
int pies_b200_tick(PiesB200Solver* s, float) { return guarded(s, [&]() { return tickOnce(s, (int)s->opt.solver, true); }); }
int pies_b200_tick_pd(PiesB200Solver* s, float) { return guarded(s, [&]() { cudaSetDevice(s->device); return pies::tickPD(s, false); }); }
int pies_b200_tick_pbd(PiesB200Solver* s, float) { return guarded(s, [&]() { cudaSetDevice(s->device); return pies::tickPBD(s, false); }); }
int pies_b200_tick_n(PiesB200Solver* s, uint32_t n) {
  return guarded(s, [&]() {
    for (uint32_t i = 0; i < n; ++i) {
      int rc = tickOnce(s, (int)s->opt.solver, i + 1 == n);
      if (rc) return rc;
    }
    return PIES_B200_OK;
  });
}
int pies_b200_set_release_hinge(PiesB200Solver* s, int r) { if (!s) return PIES_B200_EINVAL; s->releaseHinge = r != 0; return 0; }
int pies_b200_get_render_state_dirty(const PiesB200Solver* s) { return s && s->renderStateDirty ? 1 : 0; }
int pies_b200_set_render_state_dirty(PiesB200Solver* s, int d) { if (!s) return PIES_B200_EINVAL; s->renderStateDirty = d != 0; return 0; }
int pies_b200_sim_failed(const PiesB200Solver* s) { return s && s->simFailed ? 1 : 0; }
int pies_b200_clear(PiesB200Solver* s) {
  return guarded(s, [&]() {
    pies::pdAbort(s);
    pies::unregisterVertexMirror(s);
    s->scene.clear();
    // nothing of the old scene may be read back any more: no device state, no stale mirror, no collision lists
    s->deviceNewer = false; s->mirrorStale = false; s->hostStateDirty = false; s->n = 0;
    s->builtVersion = ~0ull;
    s->stats.triCollisions = s->stats.staticCollisions = 0;
    s->stats.collisionProjections = 0;
    s->colliderSet.clear(); s->colMaskColliders = 0;
    s->dragCount = 0;
    pies::clearForces(s);
    s->renderStateDirty = true;
    return PIES_B200_OK;
  });
}

// ---- render interop ----
int pies_b200_set_vertex_buffer(PiesB200Solver* s, void* deviceBuffer) {
  return guarded(s, [&]() {
    if (deviceBuffer) {
      cudaPointerAttributes attr{};
      if (cudaPointerGetAttributes(&attr, deviceBuffer) != cudaSuccess || (attr.type != cudaMemoryTypeDevice && attr.type != cudaMemoryTypeManaged)) {
        cudaGetLastError();
        return fail(s, PIES_B200_EINVAL, "set_vertex_buffer: not a device pointer");
      }
    }
    s->vtxExternal = static_cast<float*>(deviceBuffer);
    s->vtxDevValid = false;
    return PIES_B200_OK;
  });
}
int pies_b200_device_vertices(PiesB200Solver* s, void** deviceVertices, uint32_t* count) {
  if (!s || !deviceVertices) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    int rc = pies::ensureBuilt(s);
    if (rc) return rc;
    *deviceVertices = nullptr;
    if (count) *count = s->n;
    if (!s->n) return PIES_B200_OK;
    float* dev = nullptr;
    if ((rc = pies::refreshDeviceVertices(s, &dev))) return rc;
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));  // the array is complete when this returns (any stream may read it)
    *deviceVertices = dev;
    return PIES_B200_OK;
  });
}

// ---- multi-GPU halo (halo.cu) ----
int pies_b200_halo_unique_id(void* out128) {
  if (!out128) return PIES_B200_EINVAL;
  std::string err;
  int rc = pies::haloUniqueId(out128, &err);
  if (rc) g_createError = "halo_unique_id: " + err;
  return rc;
}
int pies_b200_halo_init(PiesB200Solver* s, int rank, int world, const void* id128) {
  return guarded(s, [&]() { cudaSetDevice(s->device); return pies::haloInit(s, rank, world, id128); });
}
int pies_b200_halo_set_lists(PiesB200Solver* s, int nPeers, const int* peers, const uint32_t* sendCounts, const uint32_t* sendIdx,
                             const uint32_t* recvCounts, const uint32_t* recvIdx) {
  return guarded(s, [&]() { cudaSetDevice(s->device); return pies::haloSetLists(s, nPeers, peers, sendCounts, sendIdx, recvCounts, recvIdx); });
}
int pies_b200_halo_exchange(PiesB200Solver* s, int planes) {
  return guarded(s, [&]() { cudaSetDevice(s->device); int rc = pies::haloExchange(s, planes); if (!rc) s->deviceNewer = true; return rc; });
}
int pies_b200_halo_destroy(PiesB200Solver* s) {
  return guarded(s, [&]() { cudaSetDevice(s->device); cudaStreamSynchronize(s->stream); pies::haloDestroy(s); return PIES_B200_OK; });
}

// ---- readback ----
uint32_t pies_b200_vertex_count(const PiesB200Solver* s) { return s ? (uint32_t)s->scene.vertices.size() : 0; }
uint32_t pies_b200_line_index_count(const PiesB200Solver* s) { return s ? (uint32_t)s->scene.lines.size() : 0; }
uint32_t pies_b200_triangle_count(const PiesB200Solver* s) { return s ? s->scene.triCount() : 0; }
const PiesB200Vertex* pies_b200_get_vertices(const PiesB200Solver* cs) {
  if (!cs) return nullptr;
  PiesB200Solver* s = const_cast<PiesB200Solver*>(cs);
  // The reference refreshes its mirror at the end of every substep (Solver.cpp:157,393); here the D2H copy
  // is deferred to the first getVertices() after a tick, which is observably the same and free for hosts
  // that do not read every tick.
  if (s->mirrorStale && !s->simFailed && s->builtVersion == s->scene.topologyVersion && s->n == s->scene.nodeCount()) {
    cudaSetDevice(s->device);
    pies::g_allocStream = s->stream;
    if (pies::refreshVertexMirror(s) != 0) return nullptr;
  }
  return s->scene.vertices.data();
}
const uint32_t* pies_b200_get_lines(const PiesB200Solver* s) { return s ? s->scene.lines.data() : nullptr; }
const uint32_t* pies_b200_get_triangles(const PiesB200Solver* s) { return s ? s->scene.triangles.data() : nullptr; }

// ---- reference factories ----
int pies_b200_add_nodes(PiesB200Solver* s, uint32_t n, const float* xyz) {
  if (n && !xyz) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.addNodes(n, xyz); });
}
int pies_b200_create_box(PiesB200Solver* s, const float t[3], float scale, float w) {
  if (!t) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createBox(t, scale, w); });
}
int pies_b200_create_tet_box(PiesB200Solver* s, const float t[3], float scale, const float v0[3], float w, float mass, int hinged) {
  if (!t || !v0) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createTetBox(t, scale, v0, w, mass, hinged != 0); });
}
int pies_b200_create_sheet(PiesB200Solver* s, const float t[3], float scale, float mass, float k) {
  if (!t) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createSheet(t, scale, mass, k); });
}
int pies_b200_create_shape_matching_box(PiesB200Solver* s, const float t[3], uint32_t cx, uint32_t cy, uint32_t cz, float scale,
                                        const float v0[3], float w) {
  if (!t || !cx || !cy || !cz) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createShapeMatchingBox(t, cx, cy, cz, scale, v0, w); });
}
int pies_b200_create_shape_matching_sheet(PiesB200Solver* s, const float t[3], float scale, const float v0[3], float w) {
  if (!t) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createShapeMatchingSheet(t, scale, v0, w); });
}
int pies_b200_create_bend_sheet(PiesB200Solver* s, const float t[3], float scale, float w) {
  if (!t) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.createBendSheet(t, scale, w); });
}
int pies_b200_add_tet_mesh_volume(PiesB200Solver* s, uint32_t nPoints, const float* xyz, uint32_t nTets, const uint32_t* tetIdx,
                                  uint32_t nTris, const uint32_t* triIdx, const float v0[3], float density, float strainStiffness,
                                  float minStrain, float maxStrain, float volumeStiffness, float compression, float stretching) {
  if (!s || (nPoints && !xyz) || (nTets && !tetIdx) || (nTris && !triIdx) || !v0) return PIES_B200_EINVAL;
  for (uint64_t i = 0; i < 4ull * nTets; ++i) if (tetIdx[i] >= nPoints) return fail(s, PIES_B200_EINVAL, "tet index out of range");
  for (uint64_t i = 0; i < 3ull * nTris; ++i) if (triIdx[i] >= nPoints) return fail(s, PIES_B200_EINVAL, "triangle index out of range");
  return mutate(s, [&]() {
    s->scene.addTetMeshVolume(nPoints, xyz, nTets, tetIdx, nTris, triIdx, v0, density, strainStiffness, minStrain, maxStrain,
                              volumeStiffness, compression, stretching);
  });
}
int pies_b200_add_fixed_regions(PiesB200Solver* s, uint32_t n, const float* mats, float w) {
  if (n && !mats) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.addFixedRegions(n, mats, w); });
}
int pies_b200_update_fixed_regions(PiesB200Solver* s, uint32_t n, const float* mats) {
  if (!s || (n && !mats)) return PIES_B200_EINVAL;
  // the reference asserts and returns on a count mismatch (PrimitiveUtilities.cpp:115-118)
  return guarded(s, [&]() { return s->scene.updateFixedRegions(n, mats) ? PIES_B200_OK : fail(s, PIES_B200_EINVAL, "region count mismatch"); });
}
int pies_b200_add_linked_regions(PiesB200Solver* s, uint32_t n, const float* mats, float w) {
  if (n && !mats) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.addLinkedRegions(n, mats, w); });
}

// ---- additive bulk builders ----
int pies_b200_append_nodes(PiesB200Solver* s, uint32_t n, const float* pos, const float* vel, const float* radius,
                           const float* invMass, uint32_t* firstId) {
  if (!s || (n && (!pos || !radius || !invMass))) return PIES_B200_EINVAL;
  return mutate(s, [&]() {
    size_t first = s->scene.nodeCount();
    if (firstId) *firstId = (uint32_t)first;
    const float zero[3] = {0, 0, 0};
    for (uint32_t i = 0; i < n; ++i) s->scene.appendNode(pos + 3 * i, vel ? vel + 3 * i : zero, radius[i], invMass[i]);
    s->scene.vertices.resize(s->scene.nodeCount());
    for (size_t i = first; i < s->scene.vertices.size(); ++i) {
      PiesB200Vertex& v = s->scene.vertices[i];
      std::memset(&v, 0, sizeof(v));
      std::memcpy(v.position, &s->scene.pos[3 * i], 12);
      v.radius = s->scene.radius[i];
    }
  });
}
int pies_b200_append_distance_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w) {
  if (!s || (n && !ids) || !validIds(s, ids, 2ull * n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { for (uint32_t i = 0; i < n; ++i) s->scene.appendDistance(ids[2 * i], ids[2 * i + 1], w); });
}
int pies_b200_append_position_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w) {
  if (!s || (n && !ids) || !validIds(s, ids, n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { for (uint32_t i = 0; i < n; ++i) s->scene.appendPosition(ids[i], w); });
}
int pies_b200_append_tet_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w, float lo, float hi) {
  if (!s || (n && !ids) || !validIds(s, ids, 4ull * n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { for (uint32_t i = 0; i < n; ++i) s->scene.appendTet(ids + 4 * i, w, lo, hi); });
}
int pies_b200_append_volume_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w, float lo, float hi) {
  if (!s || (n && !ids) || !validIds(s, ids, 4ull * n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { for (uint32_t i = 0; i < n; ++i) s->scene.appendVolume(ids + 4 * i, w, lo, hi); });
}
int pies_b200_append_bend_constraints(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w) {
  if (!s || (n && !ids) || !validIds(s, ids, 4ull * n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { for (uint32_t i = 0; i < n; ++i) s->scene.appendBend(ids + 4 * i, w); });
}
int pies_b200_append_shape_constraint(PiesB200Solver* s, uint32_t n, const uint32_t* ids, float w) {
  if (!s || !n || !ids || !validIds(s, ids, n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() {
    std::vector<float> mat(3ull * n);
    for (uint32_t i = 0; i < n; ++i) std::memcpy(&mat[3 * i], &s->scene.pos[3ull * ids[i]], 12);
    s->scene.appendShape(n, ids, mat.data(), w);
  });
}
int pies_b200_append_triangles(PiesB200Solver* s, uint32_t n, const uint32_t* ids) {
  if (!s || (n && !ids) || !validIds(s, ids, 3ull * n)) return PIES_B200_EINVAL;
  return mutate(s, [&]() { s->scene.triangles.insert(s->scene.triangles.end(), ids, ids + 3ull * n); ++s->scene.topologyVersion; });
}

// ---- state access ----
static int getVec(PiesB200Solver* s, int which, float* out) {
  if (!s || !out) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    if (s->deviceNewer && s->n && s->builtVersion == s->scene.topologyVersion && s->n == s->scene.nodeCount()) {
      // the live copy is on the device: one pack kernel + one DMA straight into the caller's buffer (no detour through
      // the host scene, whose copy stays marked stale)
      pies::g_allocStream = s->stream;
      const float4* src = which == 0 ? s->q.p : which == 1 ? s->prev.p : s->vel.p;
      return pies::downloadVec3(s, src, out);
    }
    int rc = pies::downloadState(s);
    if (rc) return rc;
    const std::vector<float>& v = which == 0 ? s->scene.pos : which == 1 ? s->scene.prev : s->scene.vel;
    std::memcpy(out, v.data(), v.size() * sizeof(float));
    return PIES_B200_OK;
  });
}
int pies_b200_get_positions(PiesB200Solver* s, float* xyz) { return getVec(s, 0, xyz); }
int pies_b200_get_prev_positions(PiesB200Solver* s, float* xyz) { return getVec(s, 1, xyz); }
int pies_b200_get_velocities(PiesB200Solver* s, float* xyz) { return getVec(s, 2, xyz); }

int pies_b200_set_state(PiesB200Solver* s, const float* pos, const float* prev, const float* vel) {
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    if (s->builtVersion == s->scene.topologyVersion && s->n == s->scene.nodeCount() && !s->hostStateDirty) {
      // device state is live: copy straight into it (DMA when the caller's buffers are pinned)
      if (pos) s->mirrorStale = true;
      return pies::uploadStateArrays(s, pos, prev, vel);
    }
    int rc = pies::downloadState(s);
    if (rc) return rc;
    size_t bytes = 3ull * s->scene.nodeCount() * sizeof(float);
    if (pos) std::memcpy(s->scene.pos.data(), pos, bytes);
    if (prev) std::memcpy(s->scene.prev.data(), prev, bytes);
    if (vel) std::memcpy(s->scene.vel.data(), vel, bytes);
    if (pos) for (uint32_t i = 0; i < s->scene.nodeCount(); ++i) std::memcpy(s->scene.vertices[i].position, pos + 3 * i, 12);
    s->hostStateDirty = true;
    return PIES_B200_OK;
  });
}

int pies_b200_detect(PiesB200Solver* s) {
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    int rc = pies::ensureBuilt(s);
    if (rc) return rc;
    pies::ContactLists lists;
    rc = pies::runDetection(s, lists);
    if (rc) return rc;
    cudaStreamSynchronize(s->stream);
    return PIES_B200_OK;
  });
}
int pies_b200_set_colliders(PiesB200Solver* s, uint32_t n, const PiesB200Collider* c) {
  return guarded(s, [&]() { return pies::setColliders(s, n, c); });
}
int pies_b200_get_collider_contacts(PiesB200Solver* s, uint32_t* masks) {
  if (!s || !masks) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    const uint32_t n = s->scene.nodeCount();
    if (!s->colMaskColliders || s->n != n) { std::memset(masks, 0, (size_t)n * sizeof(uint32_t)); return PIES_B200_OK; }
    PIES_CHECK(s, cudaMemcpyAsync(masks, s->colMask.p, (size_t)n * sizeof(uint32_t), cudaMemcpyDeviceToHost, s->stream));
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));
    return PIES_B200_OK;
  });
}
int pies_b200_set_drag_targets(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* targets, const float* weights) {
  return guarded(s, [&]() { return pies::setDragTargets(s, n, nodes, targets, weights); });
}
int pies_b200_set_external_forces(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* forces) {
  return guarded(s, [&]() { return pies::setExternalForces(s, n, nodes, forces); });
}
int pies_b200_set_wind(PiesB200Solver* s, const float* velocity, float normalDrag, float tangentialDrag) {
  return guarded(s, [&]() { return pies::setWind(s, velocity, normalDrag, tangentialDrag); });
}
int pies_b200_get_external_forces(PiesB200Solver* s, float* xyz) {
  return guarded(s, [&]() { return pies::getExternalForces(s, xyz); });
}
int pies_b200_raycast(PiesB200Solver* s, uint32_t nRays, const float* origins, const float* dirs, const float* tMax,
                      int32_t* tri, float* t, float* uv) {
  return guarded(s, [&]() { return pies::raycast(s, nRays, origins, dirs, tMax, tri, t, uv); });
}
uint32_t pies_b200_tri_collision_count(const PiesB200Solver* s) { return s ? s->stats.triCollisions : 0; }
uint32_t pies_b200_static_collision_count(const PiesB200Solver* s) { return s ? s->stats.staticCollisions : 0; }
int pies_b200_get_tri_collisions(PiesB200Solver* s, uint32_t* ids) {
  if (!s || !ids) return PIES_B200_EINVAL;
  if (!s->stats.triCollisions) return PIES_B200_OK;
  if (!s->detect) return PIES_B200_EINVAL;
  PIES_CHECK(s, cudaMemcpy(ids, s->detect->triList.p, 16ull * s->stats.triCollisions, cudaMemcpyDeviceToHost));
  return PIES_B200_OK;
}
int pies_b200_get_collision_csr(PiesB200Solver* s, uint64_t* nnz, int32_t* cPtr, int32_t* cCol, float* cVal, float* cDiag) {
  if (!s || !nnz) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    const uint32_t n = s->n;
    if (s->builtVersion != s->scene.topologyVersion || n != s->scene.nodeCount())
      return fail(s, PIES_B200_EINVAL, "the scene changed since the last detection: tick or detect first");
    const bool any = s->detect && (s->stats.triCollisions || s->stats.staticCollisions);
    const bool csr = any && s->stats.triCollisions && s->detect->nUnique;
    *nnz = 0;
    if (csr) {
      uint32_t last = 0;
      PIES_CHECK(s, cudaMemcpy(&last, s->detect->cPtr.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost));
      *nnz = last;
    }
    if (cPtr) {
      if (csr) PIES_CHECK(s, cudaMemcpy(cPtr, s->detect->cPtr.p, (size_t)(n + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost));
      else std::memset(cPtr, 0, (size_t)(n + 1) * sizeof(int32_t));
    }
    if (cDiag) {
      if (any) PIES_CHECK(s, cudaMemcpy(cDiag, s->detect->cDiag.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
      else std::memset(cDiag, 0, (size_t)n * sizeof(float));
    }
    if (cCol && cVal && *nnz) {
      PIES_CHECK(s, cudaMemcpy(cCol, s->detect->cCol.p, *nnz * sizeof(int32_t), cudaMemcpyDeviceToHost));
      PIES_CHECK(s, cudaMemcpy(cVal, s->detect->cVal.p, *nnz * sizeof(float), cudaMemcpyDeviceToHost));
    }
    return PIES_B200_OK;
  });
}
int pies_b200_debug_island_trace(PiesB200Solver* s, int slot, uint32_t* out4, uint32_t cap, uint32_t* count) {
  if (!s || !count || slot < 0 || slot >= pies::kIslandLists) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    *count = 0;
    if (!s->islands || !s->islands->trace.p) return fail(s, PIES_B200_EINVAL, "island trace is off: set PIES_B200_ISLAND_TRACE before the first tick");
    const uint32_t have = s->islands->listCount[slot];
    *count = have;
    const uint32_t take = std::min(have, cap);
    if (take && out4) {
      PIES_CHECK(s, cudaStreamSynchronize(s->stream));
      PIES_CHECK(s, cudaMemcpy(out4, s->islands->trace.p + (size_t)slot * s->islands->nBodies, (size_t)take * sizeof(uint4), cudaMemcpyDeviceToHost));
    }
    return PIES_B200_OK;
  });
}
int pies_b200_get_static_collisions(PiesB200Solver* s, uint32_t* ids) {
  if (!s || !ids) return PIES_B200_EINVAL;
  if (!s->stats.staticCollisions) return PIES_B200_OK;
  if (!s->detect) return PIES_B200_EINVAL;
  PIES_CHECK(s, cudaMemcpy(ids, s->detect->floorList.p, 4ull * s->stats.staticCollisions, cudaMemcpyDeviceToHost));
  return PIES_B200_OK;
}
// The occupied cells are the runs of equal keys of the sorted (cell, triangle) table; counted on the host from a copy of
// the keys (a parity readback, not a hot path), so it does not depend on which cell-start table the detection built.
static int triOccupancyStarts(PiesB200Solver* s, std::vector<uint64_t>& keys, std::vector<uint32_t>& start) {
  pies::DetectWork& w = *s->detect;
  const uint64_t P = w.nPairs;
  keys.resize(P);
  start.clear();
  if (!P) { start.push_back(0); return PIES_B200_OK; }
  cudaSetDevice(s->device);
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  PIES_CHECK(s, cudaMemcpy(keys.data(), w.keys.p, P * 8, cudaMemcpyDeviceToHost));
  for (uint64_t j = 0; j < P; ++j) if (j == 0 || keys[j] != keys[j - 1]) start.push_back((uint32_t)j);
  start.push_back((uint32_t)P);
  return PIES_B200_OK;
}
int pies_b200_tri_occupancy_counts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers) {
  if (!s || !nCells || !nMembers) return PIES_B200_EINVAL;
  *nCells = 0; *nMembers = 0;
  if (!s->detect) return PIES_B200_OK;
  return guarded(s, [&]() {
    std::vector<uint64_t> keys;
    std::vector<uint32_t> start;
    int rc = triOccupancyStarts(s, keys, start);
    if (rc) return rc;
    *nCells = start.size() - 1;
    *nMembers = s->detect->nPairs;
    return PIES_B200_OK;
  });
}
int pies_b200_get_tri_occupancy(PiesB200Solver* s, int64_t* cells, uint32_t* counts, uint32_t* members) {
  if (!s || !s->detect) return PIES_B200_EINVAL;
  return guarded(s, [&]() {
    pies::DetectWork& w = *s->detect;
    uint64_t P = w.nPairs;
    if (!P) return PIES_B200_OK;
    std::vector<uint64_t> keys;
    std::vector<uint32_t> start;
    int rc = triOccupancyStarts(s, keys, start);
    if (rc) return rc;
    const uint32_t nCells = (uint32_t)start.size() - 1;
    PIES_CHECK(s, cudaMemcpy(members, w.vals.p, P * 4, cudaMemcpyDeviceToHost));
    int by = w.keyPack[3], bz = w.keyPack[4];
    for (uint32_t c = 0; c < nCells; ++c) {
      uint64_t k = keys[start[c]];
      cells[3 * c] = (int64_t)(k >> (by + bz)) + w.keyPack[0];
      cells[3 * c + 1] = (int64_t)((k >> bz) & ((1ull << by) - 1)) + w.keyPack[1];
      cells[3 * c + 2] = (int64_t)(k & ((1ull << bz) - 1)) + w.keyPack[2];
      counts[c] = start[c + 1] - start[c];
    }
    return PIES_B200_OK;
  });
}
// ---- tick phases + halo support for slab-partitioned hosts (DESIGN.md section 7) ----
int pies_b200_pd_tick_begin(PiesB200Solver* s) { return guarded(s, [&]() { if (s->simFailed) return PIES_B200_OK; cudaSetDevice(s->device); return pies::pdTickBegin(s); }); }
int pies_b200_pd_substep_begin(PiesB200Solver* s) { return guarded(s, [&]() { if (s->simFailed) return PIES_B200_OK; cudaSetDevice(s->device); return pies::pdSubstepBegin(s); }); }
int pies_b200_pd_iteration(PiesB200Solver* s) { return guarded(s, [&]() { if (s->simFailed) return PIES_B200_OK; cudaSetDevice(s->device); return pies::pdIteration(s); }); }
int pies_b200_pd_substep_end(PiesB200Solver* s) { return guarded(s, [&]() { if (s->simFailed) return PIES_B200_OK; cudaSetDevice(s->device); return pies::pdSubstepEnd(s); }); }
int pies_b200_pd_tick_end(PiesB200Solver* s) { return guarded(s, [&]() { if (s->simFailed) return PIES_B200_OK; cudaSetDevice(s->device); return pies::pdTickEnd(s, false); }); }
int pies_b200_device_state(PiesB200Solver* s, void** q, void** prev, void** vel, uint32_t* n) {
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    int rc = pies::ensureBuilt(s);
    if (rc) return rc;
    if (q) *q = s->q.p;
    if (prev) *prev = s->prev.p;
    if (vel) *vel = s->vel.p;
    if (n) *n = s->n;
    // the caller may write ghost-node values straight into these arrays: the host copies are stale from now on
    s->deviceNewer = true; s->mirrorStale = true;
    return PIES_B200_OK;
  });
}
int pies_b200_set_triangle_order(PiesB200Solver* s, uint32_t n, const uint32_t* order) {
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    if (!order || !n) { s->haveTriOrder = false; return PIES_B200_OK; }
    if (n != s->scene.triCount()) return pies::fail(s, PIES_B200_EINVAL, "triangle order: one entry per triangle expected");
    std::vector<uint8_t> seen(n, 0);
    for (uint32_t i = 0; i < n; ++i) {
      if (order[i] >= n || seen[order[i]]) return pies::fail(s, PIES_B200_EINVAL, "triangle order is not a permutation");
      seen[order[i]] = 1;
    }
    PIES_CHECK(s, s->triOrder.upload(order, n, s->stream));
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));
    s->haveTriOrder = true;
    return PIES_B200_OK;
  });
}
int pies_b200_set_owned_nodes(PiesB200Solver* s, uint32_t n, const uint8_t* mask) {
  return guarded(s, [&]() {
    cudaSetDevice(s->device);
    if (!mask || !n) { s->haveOwnedMask = false; return PIES_B200_OK; }
    if (n != s->scene.nodeCount()) return pies::fail(s, PIES_B200_EINVAL, "owned mask: one entry per node expected");
    PIES_CHECK(s, s->ownedMask.upload(mask, n, s->stream));
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));
    s->haveOwnedMask = true;
    return PIES_B200_OK;
  });
}
int pies_b200_count_owned_contacts(PiesB200Solver* s, uint32_t* nTri, uint32_t* nFloor) {
  if (!s || !nTri || !nFloor) return PIES_B200_EINVAL;
  return guarded(s, [&]() { cudaSetDevice(s->device); return pies::countOwnedContacts(s, nTri, nFloor); });
}
int pies_b200_detect_nodes(PiesB200Solver* s) { return guarded(s, [&]() { cudaSetDevice(s->device); return pies::pbdHashOnly(s); }); }
int pies_b200_node_occupancy_counts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers) {
  if (!s || !nCells || !nMembers) return PIES_B200_EINVAL;
  return pies::pbdOccupancyCounts(s, nCells, nMembers);
}
int pies_b200_get_node_occupancy(PiesB200Solver* s, int64_t* cells, uint32_t* counts, uint32_t* members) {
  if (!s || !cells || !counts || !members) return PIES_B200_EINVAL;
  return guarded(s, [&]() { return pies::pbdOccupancy(s, cells, counts, members); });
}
int pies_b200_get_stats(const PiesB200Solver* s, PiesB200Stats* out) {
  if (!s || !out) return PIES_B200_EINVAL;
  *out = s->stats;
  out->simFailed = s->simFailed ? 1u : 0u;
  return PIES_B200_OK;
}

}  // extern "C"

// ---- host-only probe of the sliced-ELLPACK builder (system.cpp) ----
extern "C" int pies_b200_probe_sell(uint32_t n, const int32_t* rowPtr, const int32_t* col, const float* val, uint32_t* sellPtr,
                         uint32_t* sellRow, int32_t* sellCol, float* sellVal, uint64_t* paddedNnz) {
  if (!rowPtr || !paddedNnz || (n && rowPtr[n] && (!col || !val))) return PIES_B200_EINVAL;
  try {
    std::vector<uint32_t> ptr, row;
    std::vector<int> c;
    std::vector<float> v;
    pies::buildSell(n, rowPtr, col, val, ptr, row, c, v);
    *paddedNnz = c.size();
    if (sellPtr) std::memcpy(sellPtr, ptr.data(), ptr.size() * sizeof(uint32_t));
    if (sellRow) std::memcpy(sellRow, row.data(), row.size() * sizeof(uint32_t));
    if (sellCol) std::memcpy(sellCol, c.data(), c.size() * sizeof(int));
    if (sellVal) std::memcpy(sellVal, v.data(), v.size() * sizeof(float));
    return PIES_B200_OK;
  } catch (...) {
    return PIES_B200_EINVAL;
  }
}

extern "C" int pies_b200_probe_segments(uint32_t nCmds, const float* cmds, uint32_t nMeshPoints, const float* meshPoints,
                                        uint32_t nMeshTets, const uint32_t* meshTets, uint64_t* sizes, int32_t* incPtr,
                                        uint32_t* inc, uint16_t* segSlot, uint32_t* elemIds, uint32_t* segs,
                                        uint32_t* restElems, uint32_t* restNodes) {
  if (!sizes || (nCmds && !cmds)) return PIES_B200_EINVAL;
  try {
    pies::HostScene sc;
    const float zero[3] = {0.0f, 0.0f, 0.0f};
    std::vector<float> pts;
    for (uint32_t c = 0; c < nCmds; ++c) {
      const float* m = cmds + 8ull * c;
      const float* t = m + 1;
      switch ((int)m[0]) {
        case 0: sc.createTetBox(t, m[4], zero, m[5], m[6], false); break;
        case 1: sc.createSheet(t, m[4], m[5], m[6]); break;
        case 2: sc.createShapeMatchingBox(t, (uint32_t)m[4], (uint32_t)m[5], (uint32_t)m[6], m[7], zero, 1000.0f); break;
        case 3:
          if (!meshPoints || !meshTets) return PIES_B200_EINVAL;
          pts.assign(meshPoints, meshPoints + 3ull * nMeshPoints);
          for (size_t i = 0; i < pts.size(); ++i) pts[i] += t[i % 3];
          sc.addTetMeshVolume(nMeshPoints, pts.data(), nMeshTets, meshTets, 0, nullptr, zero, 1.0f, 1000.0f, 0.8f, 1.0f,
                              1000.0f, 1.0f, 1.0f);
          break;
        default: return PIES_B200_EINVAL;
      }
    }
    pies::HostSystem y;
    pies::buildSystem(sc, 1.0f / 60.0f, y, 1);
    const uint64_t sz[7] = {y.n, y.inc.size(), y.nElems, y.segs.size() / 4, y.restElems.size(), y.restNodes.size(), y.baseTet};
    std::memcpy(sizes, sz, sizeof(sz));
    auto put = [](auto* dst, const auto& v) { if (dst) std::memcpy(dst, v.data(), v.size() * sizeof(v[0])); };
    put(incPtr, y.incPtr); put(inc, y.inc); put(segSlot, y.segSlot); put(elemIds, y.elemIds); put(segs, y.segs);
    put(restElems, y.restElems); put(restNodes, y.restNodes);
    return PIES_B200_OK;
  } catch (...) {
    return PIES_B200_EINVAL;
  }
}
