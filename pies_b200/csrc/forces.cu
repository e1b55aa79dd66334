// forces.cu — external forces in the PD and PBD ticks: per-node host forces and a uniform wind acting on the triangles;
// semantics in include/pies_b200.h and DESIGN.md section 11.
//
// The force f_i of node i is evaluated once per substep, on the substep-start positions and velocities, and joins the
// velocity update (PD, k_velocity) or the advection (PBD, k_pbd_advect) exactly where gravity acts.  Host forces only:
// those kernels read the dense per-node buffer directly (no launch).  Wind on a scene with triangles: k_wind_tri writes
// each triangle's corner share to its own slot and k_force_gather sums, per node, its host force and the slots of its
// triangles in ascending triangle order over a node -> triangle CSR: no atomics, the same bits on every run.
#include <algorithm>
#include <cmath>
#include <vector>

#include "ccd.cuh"
#include "engine.h"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// f_t / 3 of triangle t = (a, b, c) in the operation order of DESIGN.md section 11, every operation rounded on its own
// (ex::, never fused).  wind = (w, c_n).  A triangle whose fp32 normal m has |m| = 0 gets 0.
__global__ void __launch_bounds__(kThreads) k_wind_tri(uint32_t nTri, const uint32_t* __restrict__ tri,
                                                       const float4* __restrict__ q, const float4* __restrict__ vel,
                                                       float4 wind, float ct, float4* __restrict__ slot) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nTri) return;
  const uint32_t a = tri[3ull * t], b = tri[3ull * t + 1], c = tri[3ull * t + 2];
  const V3 xa = v3(__ldg(q + a)), xb = v3(__ldg(q + b)), xc = v3(__ldg(q + c));
  const float4 va = __ldg(vel + a), vb = __ldg(vel + b), vc = __ldg(vel + c);
  const V3 m = ex::cross3(ex::sub(xb, xa), ex::sub(xc, xa));
  const float len = __fsqrt_rn(ex::dot3(m, m));
  float4 out = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  if (len != 0.0f) {
    const float area = ex::mul(len, 0.5f);
    const V3 nh{ex::div(m.x, len), ex::div(m.y, len), ex::div(m.z, len)};
    const V3 u{ex::sub(ex::div(ex::add(ex::add(va.x, vb.x), vc.x), 3.0f), wind.x),
               ex::sub(ex::div(ex::add(ex::add(va.y, vb.y), vc.y), 3.0f), wind.y),
               ex::sub(ex::div(ex::add(ex::add(va.z, vb.z), vc.z), 3.0f), wind.z)};
    const float un = ex::dot3(u, nh);
    const V3 ut = ex::sub(u, ex::scale(nh, un));
    const float fn = ex::mul(ex::mul(wind.w, un), fabsf(un));
    const V3 g = ex::add(ex::scale(nh, fn), ex::scale(ut, ct));
    const float na = -area;
    out = make_float4(ex::div(ex::mul(na, g.x), 3.0f), ex::div(ex::mul(na, g.y), 3.0f), ex::div(ex::mul(na, g.z), 3.0f), 0.0f);
  }
  slot[t] = out;
}

// fext[i] = host[i] (0 without host forces) + the slots of node i's triangles, added one after another in list order
// (ascending triangle index).
__global__ void __launch_bounds__(kThreads) k_force_gather(uint32_t n, const int* __restrict__ ptr,
                                                           const uint32_t* __restrict__ list, const float4* __restrict__ slot,
                                                           const float4* __restrict__ host, float4* __restrict__ fext) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 acc = host ? ldStream(host + i) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  const int beg = ptr[i], end = ptr[i + 1];
  for (int k = beg; k < end; ++k) {
    const float4 sv = __ldg(slot + list[k]);
    acc.x = ex::add(acc.x, sv.x); acc.y = ex::add(acc.y, sv.y); acc.z = ex::add(acc.z, sv.z);
  }
  acc.w = 0.0f;
  fext[i] = acc;
}

int launchForces(cudaStream_t s, uint32_t n, const ForceSet& f, const float4* q, const float4* vel) {
  if (!f.nTri || !n) return 0;
  k_wind_tri<<<gridFor(f.nTri, kThreads), kThreads, 0, s>>>(f.nTri, f.tri, q, vel, f.wind, f.ct, f.slot);
  k_force_gather<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, f.ptr, f.list, f.slot, f.host, f.fext);
  return 2;
}

// ---- host side ----------------------------------------------------------------------------------------------------
int setExternalForces(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* forces) {
  if (s->pdCtx) return fail(s, PIES_B200_EINVAL, "set_external_forces between pd_tick_begin and pd_tick_end");
  if (n && (!nodes || !forces)) return fail(s, PIES_B200_EINVAL, "set_external_forces: null array");
  const uint32_t nNodes = s->scene.nodeCount();
  std::vector<uint32_t> ids(nodes, nodes + n);
  std::vector<float4> f(n);
  for (uint32_t k = 0; k < n; ++k) {
    if (ids[k] >= nNodes) return fail(s, PIES_B200_EINVAL, "set_external_forces: node id out of range");
    const float x = forces[3ull * k], y = forces[3ull * k + 1], z = forces[3ull * k + 2];
    if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z))
      return fail(s, PIES_B200_EINVAL, "set_external_forces: non-finite force");
    f[k] = make_float4(x, y, z, 0.0f);
  }
  {
    std::vector<uint32_t> sorted(ids);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
      return fail(s, PIES_B200_EINVAL, "set_external_forces: duplicate node id");
  }
  s->forceIds.swap(ids);
  s->forceVals.swap(f);
  s->forceDirty = true;
  return PIES_B200_OK;
}

int setWind(PiesB200Solver* s, const float* velocity, float normalDrag, float tangentialDrag) {
  if (s->pdCtx) return fail(s, PIES_B200_EINVAL, "set_wind between pd_tick_begin and pd_tick_end");
  if (!velocity) return fail(s, PIES_B200_EINVAL, "set_wind: null velocity");
  for (int a = 0; a < 3; ++a)
    if (!std::isfinite(velocity[a])) return fail(s, PIES_B200_EINVAL, "set_wind: non-finite velocity");
  if (!std::isfinite(normalDrag) || !std::isfinite(tangentialDrag))
    return fail(s, PIES_B200_EINVAL, "set_wind: non-finite drag coefficient");
  if (normalDrag < 0.0f || tangentialDrag < 0.0f) return fail(s, PIES_B200_EINVAL, "set_wind: negative drag coefficient");
  s->wind = make_float4(velocity[0], velocity[1], velocity[2], normalDrag);
  s->windTangential = tangentialDrag;
  return PIES_B200_OK;
}

// At the start of a tick, after ensureBuilt: brings the dense host-force buffer and the wind's node -> triangle CSR up to
// date with the current sets and topology, and fixes which of them the tick applies (forceSet).
int prepareForces(PiesB200Solver* s) {
  const uint32_t n = s->n;
  cudaStream_t st = s->stream;
  const bool host = !s->forceIds.empty();
  const uint32_t nTri = s->scene.triCount();
  const bool wind = (s->wind.w != 0.0f || s->windTangential != 0.0f) && nTri && n;
  if (host && (s->forceDirty || s->forceDenseN != n)) {
    std::vector<float4> dense(n, make_float4(0.0f, 0.0f, 0.0f, 0.0f));
    for (size_t k = 0; k < s->forceIds.size(); ++k) dense[s->forceIds[k]] = s->forceVals[k];
    PIES_CHECK(s, s->hostForce.upload(dense.data(), n, st));
    PIES_CHECK(s, cudaStreamSynchronize(st));   // the staging vector dies here
    s->forceDirty = false;
    s->forceDenseN = n;
  }
  if (wind && s->windCsrVersion != s->scene.topologyVersion) {
    // counting sort of the corners by node; triangles are visited in ascending order, so each node's list is ascending
    const std::vector<uint32_t>& tri = s->scene.triangles;
    std::vector<int> ptr(n + 1, 0);
    for (uint32_t id : tri) ++ptr[id + 1];
    for (uint32_t i = 0; i < n; ++i) ptr[i + 1] += ptr[i];
    std::vector<int> next(ptr.begin(), ptr.end() - 1);
    std::vector<uint32_t> list(tri.size());
    for (size_t k = 0; k < tri.size(); ++k) list[next[tri[k]]++] = (uint32_t)(k / 3);
    PIES_CHECK(s, s->windPtr.upload(ptr.data(), ptr.size(), st));
    PIES_CHECK(s, s->windList.upload(list.data(), list.size(), st));
    PIES_CHECK(s, s->windSlot.reserve(nTri));
    PIES_CHECK(s, s->fext.reserve(n));
    PIES_CHECK(s, cudaStreamSynchronize(st));
    s->windCsrVersion = s->scene.topologyVersion;
  }
  s->forceMode = (host ? 1u : 0u) | (wind ? 2u : 0u);
  s->forceModeN = n;
  return PIES_B200_OK;
}

int getExternalForces(PiesB200Solver* s, float* xyz) {
  if (!xyz) return fail(s, PIES_B200_EINVAL, "get_external_forces: null array");
  const uint32_t nNodes = s->scene.nodeCount();
  std::fill(xyz, xyz + 3ull * nNodes, 0.0f);
  const float4* src = forceSet(s).field();
  const uint32_t n = std::min(s->forceModeN, nNodes);
  if (!src || !n) return PIES_B200_OK;
  std::vector<float4> f(n);
  PIES_CHECK(s, cudaMemcpyAsync(f.data(), src, (size_t)n * sizeof(float4), cudaMemcpyDeviceToHost, s->stream));
  PIES_CHECK(s, cudaStreamSynchronize(s->stream));
  for (uint32_t i = 0; i < n; ++i) { xyz[3ull * i] = f[i].x; xyz[3ull * i + 1] = f[i].y; xyz[3ull * i + 2] = f[i].z; }
  return PIES_B200_OK;
}

void clearForces(PiesB200Solver* s) {
  s->forceIds.clear(); s->forceVals.clear();
  s->forceDirty = false; s->forceDenseN = 0;
  s->wind = make_float4(0.0f, 0.0f, 0.0f, 0.0f); s->windTangential = 0.0f;
  s->windCsrVersion = ~0ull;
  s->windPtr.release(); s->windList.release(); s->windSlot.release(); s->fext.release();
  s->forceMode = 0; s->forceModeN = 0;
}

}  // namespace pies
