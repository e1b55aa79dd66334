// colliders.cu — static colliders (half-spaces, spheres, oriented boxes) in the PD and PBD ticks; semantics in
// include/pies_b200.h and DESIGN.md section 9.
//
// A PD node-collider contact is a one-node constraint of weight 1e4, like the floor's StaticCollisionConstraint: it
// adds to the per-node diagonal (floorW -> cDiag) and one projected target per iteration to the right-hand side, so
// islands, segments and the C_t CSR keep their structure.  Every kernel here stages the solver's colliders (at most
// 32, 2 KB) in shared memory and walks a node's colliders in ascending index order.
#include <cmath>
#include <vector>

#include "collider.cuh"
#include "engine.h"
#include "rhs.cuh"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- detection (once per substep, on the predicted positions): mask + the diagonal weight after the floor's ----------
__global__ void __launch_bounds__(kThreads) k_collider_detect(uint32_t n, const PiesB200Collider* __restrict__ col, uint32_t nCol,
                                                              const float4* __restrict__ q, float thickness, int haveFloor,
                                                              uint32_t* __restrict__ mask, float* __restrict__ floorW) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = q[i];
  float w = haveFloor ? floorW[i] : 0.0f;
  uint32_t m = 0;
  for (uint32_t k = 0; k < nCol; ++k) {
    float3 nrm;
    if (colliderPhi(sCol[k], p.x, p.y, p.z, &nrm) < thickness) { m |= 1u << k; w += kFloorW; }
  }
  mask[i] = m;
  floorW[i] = w;
}

// ---- local step: sum of the weighted projections, formed once per node (addContactTerms adds it) -------------------
__global__ void __launch_bounds__(kThreads) k_collider_project(uint32_t n, const PiesB200Collider* __restrict__ col, uint32_t nCol,
                                                               const uint32_t* __restrict__ mask, const float4* __restrict__ q,
                                                               float4* __restrict__ colRhs) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t m = mask[i];
  if (!m) return;
  const float4 p = q[i];
  float4 acc = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  for (; m; m &= m - 1) {
    const float3 t = colliderProject(sCol[__ffs(m) - 1], make_float3(p.x, p.y, p.z));
    acc.x += kFloorW * t.x; acc.y += kFloorW * t.y; acc.z += kFloorW * t.z;
  }
  colRhs[i] = acc;
}

// ---- after stabilisation: each contact's projection in sequence, from the current position (only q moves) ----------
__global__ void __launch_bounds__(kThreads) k_collider_snap(uint32_t n, const PiesB200Collider* __restrict__ col, uint32_t nCol,
                                                            const uint32_t* __restrict__ mask, float4* __restrict__ q) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t m = mask[i];
  if (!m) return;
  const float4 p = q[i];
  float3 x = make_float3(p.x, p.y, p.z);
  for (; m; m &= m - 1) x = colliderProject(sCol[__ffs(m) - 1], x);
  q[i] = make_float4(x.x, x.y, x.z, p.w);
}

// ---- friction: k_floor_friction's rule in the tangent plane of each contact (with n = +y it is that kernel) ---------
__global__ void __launch_bounds__(kThreads) k_collider_friction(uint32_t n, const PiesB200Collider* __restrict__ col, uint32_t nCol,
                                                                const uint32_t* __restrict__ mask, const float4* __restrict__ q,
                                                                float4* __restrict__ vel, float friction, float staticThreshold) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t m = mask[i];
  if (!m) return;
  const float4 p = q[i];
  float4 v = vel[i];
  for (; m; m &= m - 1) {
    float3 nr;
    colliderPhi(sCol[__ffs(m) - 1], p.x, p.y, p.z, &nr);
    const float vn = v.x * nr.x + v.y * nr.y + v.z * nr.z;
    const float tx = v.x - vn * nr.x, ty = v.y - vn * nr.y, tz = v.z - vn * nr.z;
    const float fr = sqrtf(tx * tx + ty * ty + tz * tz) < staticThreshold ? 1.0f : friction;
    v.x += (-fr) * tx; v.y += (-fr) * ty; v.z += (-fr) * tz;
  }
  vel[i] = v;
}

// ---- PBD (radius = prev.w): clamp to phi = r after the floor clamp, friction after the velocity update --------------
__global__ void __launch_bounds__(kThreads) k_pbd_collider_clamp(uint32_t n, const PiesB200Collider* __restrict__ col, uint32_t nCol,
                                                                 float4* __restrict__ q, const float4* __restrict__ prev) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i];
  const float r = prev[i].w;
  bool moved = false;
  for (uint32_t k = 0; k < nCol; ++k) {
    float3 nr;
    const float phi = colliderPhi(sCol[k], p.x, p.y, p.z, &nr);
    if (phi - r < 0.0f) {
      const float d = r - phi;
      p.x += d * nr.x; p.y += d * nr.y; p.z += d * nr.z;
      moved = true;
    }
  }
  if (moved) q[i] = p;
}

// the floor's rule (pbd.cu, k_pbd_velocity): planar speed below 5 stops, otherwise it is scaled by 1 - friction
__global__ void __launch_bounds__(kThreads) k_pbd_collider_friction(uint32_t n, const PiesB200Collider* __restrict__ col,
                                                                    uint32_t nCol, const float4* __restrict__ q,
                                                                    const float4* __restrict__ prev, float4* __restrict__ vel,
                                                                    float friction) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float4 p = q[i];
  const float r = prev[i].w;
  float4 v = vel[i];
  bool touched = false;
  for (uint32_t k = 0; k < nCol; ++k) {
    float3 nr;
    if (colliderPhi(sCol[k], p.x, p.y, p.z, &nr) - r > 0.0f) continue;
    const float vn = v.x * nr.x + v.y * nr.y + v.z * nr.z;
    const float tx = v.x - vn * nr.x, ty = v.y - vn * nr.y, tz = v.z - vn * nr.z;
    const float f = sqrtf(tx * tx + ty * ty + tz * tz) < 5.0f ? 0.0f : 1.0f - friction;
    v.x = vn * nr.x + f * tx; v.y = vn * nr.y + f * ty; v.z = vn * nr.z + f * tz;
    touched = true;
  }
  if (touched) vel[i] = v;
}

int launchColliderDetect(cudaStream_t s, uint32_t n, const ColliderSet& c, const float4* q, float thickness, bool haveFloor,
                         uint32_t* mask, float* floorW) {
  if (!n || !c.n) return 0;
  k_collider_detect<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, q, thickness, haveFloor ? 1 : 0, mask, floorW);
  return 1;
}

int launchColliderProject(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, const float4* q, float4* colRhs) {
  if (!n || !c.n) return 0;
  k_collider_project<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, mask, q, colRhs);
  return 1;
}

int launchColliderSnap(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, float4* q) {
  if (!n || !c.n) return 0;
  k_collider_snap<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, mask, q);
  return 1;
}

int launchColliderFriction(cudaStream_t s, uint32_t n, const ColliderSet& c, const uint32_t* mask, const float4* q, float4* vel,
                           float friction, float staticThreshold) {
  if (!n || !c.n) return 0;
  k_collider_friction<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, mask, q, vel, friction, staticThreshold);
  return 1;
}

int launchPbdColliderClamp(cudaStream_t s, uint32_t n, const ColliderSet& c, float4* q, const float4* prev) {
  if (!n || !c.n) return 0;
  k_pbd_collider_clamp<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, q, prev);
  return 1;
}

int launchPbdColliderFriction(cudaStream_t s, uint32_t n, const ColliderSet& c, const float4* q, const float4* prev, float4* vel,
                              float friction) {
  if (!n || !c.n) return 0;
  k_pbd_collider_friction<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.col, c.n, q, prev, vel, friction);
  return 1;
}

// ---- host: validation of a caller's set (set_colliders and the probe) -----------------------------------------------
int prepareColliders(uint32_t n, const PiesB200Collider* in, std::vector<PiesB200Collider>& out, const char** why) {
  if (n > kMaxColliders) { *why = "more than 32 colliders (the width of the per-node contact mask)"; return PIES_B200_ERANGE; }
  if (n && !in) { *why = "null collider array"; return PIES_B200_EINVAL; }
  out.assign(in, in + n);
  for (PiesB200Collider& c : out) {
    const float* f = c.center;  // center, axes, extent: 15 consecutive floats
    for (int k = 0; k < 15; ++k)
      if (!std::isfinite(f[k])) { *why = "non-finite collider value"; return PIES_B200_EINVAL; }
    if (c.kind == PIES_B200_COLLIDER_HALFSPACE) {
      const double x = c.axes[0], y = c.axes[1], z = c.axes[2], len = std::sqrt(x * x + y * y + z * z);
      if (!(len > 0.0) || !std::isfinite(len)) { *why = "half-space with a zero normal"; return PIES_B200_EINVAL; }
      c.axes[0] = (float)(x / len); c.axes[1] = (float)(y / len); c.axes[2] = (float)(z / len);
    } else if (c.kind == PIES_B200_COLLIDER_SPHERE) {
      if (!(c.extent[0] > 0.0f)) { *why = "sphere radius <= 0"; return PIES_B200_EINVAL; }
    } else if (c.kind == PIES_B200_COLLIDER_BOX) {
      for (int a = 0; a < 3; ++a)
        if (!(c.extent[a] > 0.0f)) { *why = "box half extent <= 0"; return PIES_B200_EINVAL; }
      for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) {
          const double d = (double)c.axes[3 * a] * c.axes[3 * b] + (double)c.axes[3 * a + 1] * c.axes[3 * b + 1] +
                           (double)c.axes[3 * a + 2] * c.axes[3 * b + 2];
          if (std::fabs(d - (a == b ? 1.0 : 0.0)) > 1e-4) { *why = "box axes are not orthonormal within 1e-4"; return PIES_B200_EINVAL; }
        }
    } else {
      *why = "unknown collider kind"; return PIES_B200_EINVAL;
    }
  }
  return PIES_B200_OK;
}

int setColliders(PiesB200Solver* s, uint32_t n, const PiesB200Collider* c) {
  // the masks of a substep index the set it was detected with
  if (s->pdCtx) return fail(s, PIES_B200_EINVAL, "set_colliders between pd_tick_begin and pd_tick_end");
  std::vector<PiesB200Collider> set;
  const char* why = nullptr;
  const int rc = prepareColliders(n, c, set, &why);
  if (rc) return fail(s, rc, why);
  if (!set.empty()) {
    PIES_CHECK(s, s->colliders.upload(set.data(), set.size(), s->stream));
    PIES_CHECK(s, cudaStreamSynchronize(s->stream));   // the staging vector dies here
  }
  s->colliderSet.swap(set);
  return PIES_B200_OK;
}

__global__ void k_probe_colliders(uint32_t nPts, const float* __restrict__ xyz, const PiesB200Collider* __restrict__ col,
                                  uint32_t nCol, float* __restrict__ phi, float* __restrict__ nrm) {
  __shared__ PiesB200Collider sCol[kMaxColliders];
  stageColliders(sCol, col, nCol);
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nPts) return;
  for (uint32_t k = 0; k < nCol; ++k) {
    float3 nr;
    const uint64_t o = (uint64_t)i * nCol + k;
    phi[o] = colliderPhi(sCol[k], xyz[3ull * i], xyz[3ull * i + 1], xyz[3ull * i + 2], &nr);
    nrm[3 * o] = nr.x; nrm[3 * o + 1] = nr.y; nrm[3 * o + 2] = nr.z;
  }
}

void preloadColliderKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_collider_detect);
  cudaFuncGetAttributes(&a, k_collider_project);
  cudaFuncGetAttributes(&a, k_collider_snap);
  cudaFuncGetAttributes(&a, k_collider_friction);
}

}  // namespace pies

extern "C" int pies_b200_probe_colliders(uint32_t nPoints, const float* xyz, uint32_t nColliders, const PiesB200Collider* c,
                                         float* phi, float* normals) {
  using namespace pies;
  std::vector<PiesB200Collider> set;
  const char* why = nullptr;
  int rc = prepareColliders(nColliders, c, set, &why);
  if (rc) return rc;
  if (!nPoints || !nColliders) return PIES_B200_OK;
  if (!xyz || !phi || !normals) return PIES_B200_EINVAL;
  int dev = 0;
  if (cudaGetDeviceCount(&dev) != cudaSuccess || dev == 0) { cudaGetLastError(); return PIES_B200_ENODEV; }
  const size_t nOut = (size_t)nPoints * nColliders;
  float *dx = nullptr, *dphi = nullptr, *dn = nullptr;
  PiesB200Collider* dc = nullptr;
  cudaError_t e = cudaMalloc(&dx, 12ull * nPoints);
  if (e == cudaSuccess) e = cudaMalloc(&dc, sizeof(PiesB200Collider) * nColliders);
  if (e == cudaSuccess) e = cudaMalloc(&dphi, 4 * nOut);
  if (e == cudaSuccess) e = cudaMalloc(&dn, 12 * nOut);
  if (e == cudaSuccess) e = cudaMemcpy(dx, xyz, 12ull * nPoints, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemcpy(dc, set.data(), sizeof(PiesB200Collider) * nColliders, cudaMemcpyHostToDevice);
  if (e == cudaSuccess) {
    k_probe_colliders<<<gridFor(nPoints, kThreads), kThreads>>>(nPoints, dx, dc, nColliders, dphi, dn);
    e = cudaDeviceSynchronize();
  }
  if (e == cudaSuccess) e = cudaMemcpy(phi, dphi, 4 * nOut, cudaMemcpyDeviceToHost);
  if (e == cudaSuccess) e = cudaMemcpy(normals, dn, 12 * nOut, cudaMemcpyDeviceToHost);
  cudaFree(dx); cudaFree(dc); cudaFree(dphi); cudaFree(dn);
  if (e != cudaSuccess) { cudaGetLastError(); return PIES_B200_ECUDA; }
  return PIES_B200_OK;
}
