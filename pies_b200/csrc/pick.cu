// pick.cu — drag targets in the PD and PBD ticks, and the ray query an interactive host picks with; semantics in
// include/pies_b200.h and DESIGN.md section 10.
//
// A drag is a one-node position constraint (A = B = [1]) whose target and weight the host replaces between ticks.  In
// PD its weight joins the per-node diagonal the floor and the colliders already use (floorW -> cDiag), so islands,
// segments and the C_t CSR keep their structure, and w g is constant for the substep, so it goes into msn (the base of
// every right-hand side) once per substep instead of into the per-iteration kernels.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <limits>
#include <vector>

#include "ccd.cuh"
#include "engine.h"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- drags ------------------------------------------------------------------------------------------------------
// PD detection, after k_floor_weight / k_collider_detect and before k_ccsr_fill: the drag's weight after the floor's
// and the colliders', and w g into msn = M s_n / h^2 (written by k_predict this substep, read only by the RHS kernels).
// Ids are unique, so no two threads touch one node.
__global__ void __launch_bounds__(kThreads) k_drag_terms(uint32_t n, const uint32_t* __restrict__ node,
                                                         const float4* __restrict__ targetW, float* __restrict__ floorW,
                                                         float4* __restrict__ msn) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = node[k];
  const float4 g = targetW[k];
  floorW[i] += g.w;
  float4 m = msn[i];
  m.x += g.w * g.x; m.y += g.w * g.y; m.z += g.w * g.z;
  msn[i] = m;
}

// PBD: PosOp's rule (pbd.cu) with the weight clamped to 1, so a PD-sized weight puts the node on its target
__global__ void __launch_bounds__(kThreads) k_pbd_drag(uint32_t n, const uint32_t* __restrict__ node,
                                                       const float4* __restrict__ targetW, float4* __restrict__ q) {
  const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = node[k];
  const float4 g = targetW[k];
  const float w = fminf(g.w, 1.0f);
  float4 p = q[i];
  p.x = ex::add(p.x, ex::mul(w, ex::sub(g.x, p.x)));
  p.y = ex::add(p.y, ex::mul(w, ex::sub(g.y, p.y)));
  p.z = ex::add(p.z, ex::mul(w, ex::sub(g.z, p.z)));
  q[i] = p;
}

int launchDragTerms(cudaStream_t s, const DragSet& d, float* floorW, float4* msn) {
  if (!d.n) return 0;
  k_drag_terms<<<gridFor(d.n, kThreads), kThreads, 0, s>>>(d.n, d.node, d.targetW, floorW, msn);
  return 1;
}

int launchPbdDrag(cudaStream_t s, const DragSet& d, float4* q) {
  if (!d.n) return 0;
  k_pbd_drag<<<gridFor(d.n, kThreads), kThreads, 0, s>>>(d.n, d.node, d.targetW, q);
  return 1;
}

int setDragTargets(PiesB200Solver* s, uint32_t n, const uint32_t* nodes, const float* targets, const float* weights) {
  // a substep's detection added the set it saw to msn and the diagonal
  if (s->pdCtx) return fail(s, PIES_B200_EINVAL, "set_drag_targets between pd_tick_begin and pd_tick_end");
  if (n && (!nodes || !targets || !weights)) return fail(s, PIES_B200_EINVAL, "set_drag_targets: null array");
  const uint32_t nNodes = s->scene.nodeCount();
  std::vector<uint32_t> ids(nodes, nodes + n);
  std::vector<float4> tw(n);
  for (uint32_t k = 0; k < n; ++k) {
    if (ids[k] >= nNodes) return fail(s, PIES_B200_EINVAL, "set_drag_targets: node id out of range");
    const float x = targets[3ull * k], y = targets[3ull * k + 1], z = targets[3ull * k + 2], w = weights[k];
    if (!std::isfinite(x) || !std::isfinite(y) || !std::isfinite(z) || !std::isfinite(w))
      return fail(s, PIES_B200_EINVAL, "set_drag_targets: non-finite target or weight");
    if (!(w > 0.0f)) return fail(s, PIES_B200_EINVAL, "set_drag_targets: weight <= 0");
    tw[k] = make_float4(x, y, z, w);
  }
  {
    std::vector<uint32_t> sorted(ids);
    std::sort(sorted.begin(), sorted.end());
    if (std::adjacent_find(sorted.begin(), sorted.end()) != sorted.end())
      return fail(s, PIES_B200_EINVAL, "set_drag_targets: duplicate node id");
  }
  if (n) {
    PIES_CHECK(s, s->dragNode.upload(ids.data(), n, s->stream));
    PIES_CHECK(s, s->dragTargetW.upload(tw.data(), n, s->stream));
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));   // the staging vectors die here
  }
  s->dragCount = n;
  return PIES_B200_OK;
}

// ---- raycast --------------------------------------------------------------------------------------------------------
constexpr int kRayChunk = 256;   // rays staged in shared memory at a time (= the CTA size)

// Moller-Trumbore in the operation order of DESIGN.md section 10, every operation rounded on its own (ccd.cuh: ex::,
// never fused).  e1 = p1 - p0, e2 = p2 - p0; the caller has rejected a triangle with cross(e1, e2) == 0.  Returns false
// for a ray parallel to the plane (det == 0), outside the triangle or outside [0, tMax]; t is returned with -0 as +0.
__device__ __forceinline__ bool rayTriangle(const float4& o, const float4& d, V3 p0, V3 e1, V3 e2, float& t, float& u, float& v) {
  const V3 dir{d.x, d.y, d.z};
  const V3 pv = ex::cross3(dir, e2);
  const float det = ex::dot3(e1, pv);
  if (det == 0.0f) return false;
  const float inv = ex::div(1.0f, det);
  const V3 sv = ex::sub(V3{o.x, o.y, o.z}, p0);
  u = ex::mul(ex::dot3(sv, pv), inv);
  if (!(u >= 0.0f && u <= 1.0f)) return false;
  const V3 qv = ex::cross3(sv, e1);
  v = ex::mul(ex::dot3(dir, qv), inv);
  if (!(v >= 0.0f && ex::add(u, v) <= 1.0f)) return false;
  t = ex::mul(ex::dot3(e2, qv), inv);
  if (!(t >= 0.0f && t <= o.w)) return false;
  t = ex::add(t, 0.0f);   // -0 -> +0: the key below orders by the bits of t
  return true;
}

// corners of triangle f; false when it has zero area (cross(e1, e2) == 0 in fp32) and can never be hit
__device__ __forceinline__ bool triangleEdges(uint32_t f, const uint32_t* __restrict__ tri, const float4* __restrict__ q,
                                              V3& p0, V3& e1, V3& e2) {
  const float4 a = q[tri[3ull * f]], b = q[tri[3ull * f + 1]], c = q[tri[3ull * f + 2]];
  p0 = V3{a.x, a.y, a.z};
  e1 = ex::sub(V3{b.x, b.y, b.z}, p0);
  e2 = ex::sub(V3{c.x, c.y, c.z}, p0);
  const V3 nr = ex::cross3(e1, e2);
  return nr.x != 0.0f || nr.y != 0.0f || nr.z != 0.0f;
}

// One thread per triangle (grid-stride), its corners loaded once; the rays pass through shared memory in chunks of
// kRayChunk.  rays[2r] = (origin, tMax), rays[2r + 1] = (direction, 0).  A hit lowers key[r] to (bits of t) << 32 | f:
// t >= 0, so the unsigned order of the key is the order of t, then of the triangle index, whatever order threads run in.
__global__ void __launch_bounds__(kRayChunk) k_raycast(uint32_t nTri, const uint32_t* __restrict__ tri, const float4* __restrict__ q,
                                                       uint32_t nRays, const float4* __restrict__ rays,
                                                       unsigned long long* __restrict__ key) {
  __shared__ float4 sO[kRayChunk], sD[kRayChunk];
  const uint32_t stride = gridDim.x * blockDim.x;
  for (uint32_t base = blockIdx.x * blockDim.x; base < nTri; base += stride) {   // uniform over the CTA (barriers below)
    const uint32_t f = base + threadIdx.x;
    V3 p0{}, e1{}, e2{};
    const bool live = f < nTri && triangleEdges(f, tri, q, p0, e1, e2);
    for (uint32_t r0 = 0; r0 < nRays; r0 += kRayChunk) {
      const uint32_t m = min((uint32_t)kRayChunk, nRays - r0);
      __syncthreads();
      if (threadIdx.x < m) { sO[threadIdx.x] = rays[2ull * (r0 + threadIdx.x)]; sD[threadIdx.x] = rays[2ull * (r0 + threadIdx.x) + 1]; }
      __syncthreads();
      if (!live) continue;
      for (uint32_t k = 0; k < m; ++k) {
        float t, u, v;
        if (rayTriangle(sO[k], sD[k], p0, e1, e2, t, u, v))
          atomicMin(key + r0 + k, ((unsigned long long)__float_as_uint(t) << 32) | f);
      }
    }
  }
}

// Per ray: the winning triangle and t from the key, u and v recomputed for that triangle only (the same operations as
// the test that produced the key, so the same bits).  out[r] = (tri as int bits, t, u, v).
__global__ void __launch_bounds__(kThreads) k_ray_decode(uint32_t nRays, const float4* __restrict__ rays,
                                                         const unsigned long long* __restrict__ key,
                                                         const uint32_t* __restrict__ tri, const float4* __restrict__ q,
                                                         float4* __restrict__ out) {
  const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= nRays) return;
  const unsigned long long kv = key[r];
  float4 res = make_float4(__int_as_float(-1), __uint_as_float(0x7f800000u), 0.0f, 0.0f);
  if (kv != ~0ull) {
    const uint32_t f = (uint32_t)kv;
    V3 p0, e1, e2;
    triangleEdges(f, tri, q, p0, e1, e2);
    float t = 0.0f, u = 0.0f, v = 0.0f;
    rayTriangle(rays[2ull * r], rays[2ull * r + 1], p0, e1, e2, t, u, v);
    res = make_float4(__int_as_float((int)f), __uint_as_float((uint32_t)(kv >> 32)), u, v);
  }
  out[r] = res;
}

int raycast(PiesB200Solver* s, uint32_t nRays, const float* origins, const float* dirs, const float* tMax, int32_t* tri,
            float* t, float* uv) {
  if (nRays && (!origins || !dirs || !tMax || !tri || !t || !uv)) return fail(s, PIES_B200_EINVAL, "raycast: null array");
  for (uint32_t r = 0; r < nRays; ++r) {
    const float* o = origins + 3ull * r;
    const float* d = dirs + 3ull * r;
    for (int a = 0; a < 3; ++a)
      if (!std::isfinite(o[a]) || !std::isfinite(d[a])) return fail(s, PIES_B200_EINVAL, "raycast: non-finite origin or direction");
    if (d[0] == 0.0f && d[1] == 0.0f && d[2] == 0.0f) return fail(s, PIES_B200_EINVAL, "raycast: zero direction");
    if (!(tMax[r] >= 0.0f)) return fail(s, PIES_B200_EINVAL, "raycast: tMax NaN or negative");
  }
  for (uint32_t r = 0; r < nRays; ++r) {
    tri[r] = -1; t[r] = std::numeric_limits<float>::infinity(); uv[2ull * r] = uv[2ull * r + 1] = 0.0f;
  }
  if (!nRays) return PIES_B200_OK;
  int rc = ensureBuilt(s);
  if (rc) return rc;
  const uint32_t nTri = s->scene.triCount();
  if (!nTri || !s->n) return PIES_B200_OK;
  cudaStream_t st = s->stream;
  std::vector<float4> packed(2ull * nRays);
  for (uint32_t r = 0; r < nRays; ++r) {
    packed[2ull * r] = make_float4(origins[3ull * r], origins[3ull * r + 1], origins[3ull * r + 2], tMax[r]);
    packed[2ull * r + 1] = make_float4(dirs[3ull * r], dirs[3ull * r + 1], dirs[3ull * r + 2], 0.0f);
  }
  PIES_CHECK(s, s->rays.upload(packed.data(), packed.size(), st));
  PIES_CHECK(s, s->rayKey.reserve(nRays));
  PIES_CHECK(s, s->rayHit.reserve(nRays));
  PIES_CHECK(s, cudaMemsetAsync(s->rayKey.p, 0xff, (size_t)nRays * sizeof(unsigned long long), st));
  const int grid = std::min(gridFor(nTri, kRayChunk), kNumSMs * 8);
  k_raycast<<<grid, kRayChunk, 0, st>>>(nTri, s->triIds.p, s->q.p, nRays, s->rays.p, s->rayKey.p);
  k_ray_decode<<<gridFor(nRays, kThreads), kThreads, 0, st>>>(nRays, s->rays.p, s->rayKey.p, s->triIds.p, s->q.p, s->rayHit.p);
  s->launches += 2;
  std::vector<float4> hits(nRays);
  PIES_CHECK(s, cudaMemcpyAsync(hits.data(), s->rayHit.p, (size_t)nRays * sizeof(float4), cudaMemcpyDeviceToHost, st));
  PIES_CHECK(s, cudaStreamSynchronize(st));   // also keeps `packed` alive until the upload has been read
  for (uint32_t r = 0; r < nRays; ++r) {
    int32_t f;
    std::memcpy(&f, &hits[r].x, sizeof(f));
    tri[r] = f; t[r] = hits[r].y; uv[2ull * r] = hits[r].z; uv[2ull * r + 1] = hits[r].w;
  }
  return PIES_B200_OK;
}

}  // namespace pies
