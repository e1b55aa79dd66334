// collider.cuh — signed distance and outward normal of the static colliders (include/pies_b200.h, DESIGN.md section 9),
// shared by the PD and PBD collider kernels (colliders.cu) and the probe.
#pragma once

#include "../../include/pies_b200.h"
#include "common.cuh"

namespace pies {

constexpr uint32_t kMaxColliders = PIES_B200_MAX_COLLIDERS;
constexpr uint32_t kColliderWords = sizeof(PiesB200Collider) / 4;
static_assert(sizeof(PiesB200Collider) == 64, "PiesB200Collider is 64 bytes");

// Copies the n colliders of a solver into shared memory (all threads of the CTA take part; ends with a barrier).
__device__ __forceinline__ void stageColliders(PiesB200Collider* dst, const PiesB200Collider* __restrict__ src, uint32_t n) {
  const uint32_t* s = reinterpret_cast<const uint32_t*>(src);
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  for (uint32_t t = threadIdx.x; t < n * kColliderWords; t += blockDim.x) d[t] = __ldg(s + t);
  __syncthreads();
}

// phi(x) of collider c; *nrm receives n(x).
__device__ __forceinline__ float colliderPhi(const PiesB200Collider& c, float x, float y, float z, float3* nrm) {
  const float dx = x - c.center[0], dy = y - c.center[1], dz = z - c.center[2];
  if (c.kind == PIES_B200_COLLIDER_HALFSPACE) {
    *nrm = make_float3(c.axes[0], c.axes[1], c.axes[2]);
    return c.axes[0] * dx + c.axes[1] * dy + c.axes[2] * dz;
  }
  if (c.kind == PIES_B200_COLLIDER_SPHERE) {
    const float len = sqrtf(dx * dx + dy * dy + dz * dz);
    *nrm = len > 0.0f ? make_float3(dx / len, dy / len, dz / len) : make_float3(0.0f, 1.0f, 0.0f);
    return len - c.extent[0];
  }
  // box: local coordinates d_a = axis_a . (x - c), q_a = |d_a| - e_a
  float d[3], q[3];
  bool outside = false;
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    d[a] = c.axes[3 * a] * dx + c.axes[3 * a + 1] * dy + c.axes[3 * a + 2] * dz;
    q[a] = fabsf(d[a]) - c.extent[a];
    outside = outside || q[a] > 0.0f;
  }
  if (outside) {  // closest surface point to x, in local coordinates o = sign(d) max(q, 0)
    float o[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) o[a] = q[a] > 0.0f ? (d[a] < 0.0f ? -q[a] : q[a]) : 0.0f;
    const float len = sqrtf(o[0] * o[0] + o[1] * o[1] + o[2] * o[2]);
    const float u0 = o[0] / len, u1 = o[1] / len, u2 = o[2] / len;
    *nrm = make_float3(u0 * c.axes[0] + u1 * c.axes[3] + u2 * c.axes[6], u0 * c.axes[1] + u1 * c.axes[4] + u2 * c.axes[7],
                       u0 * c.axes[2] + u1 * c.axes[5] + u2 * c.axes[8]);
    return len;
  }
  int a = 0;  // nearest face: largest q, the lowest axis on a tie, the + side when d_a = 0
  if (q[1] > q[a]) a = 1;
  if (q[2] > q[a]) a = 2;
  const float sgn = d[a] < 0.0f ? -1.0f : 1.0f;
  *nrm = make_float3(sgn * c.axes[3 * a], sgn * c.axes[3 * a + 1], sgn * c.axes[3 * a + 2]);
  return q[a];
}

// PD projection onto collider c: p = x - min(phi(x), 0) n(x) (only a penetrating point moves, onto the surface).
__device__ __forceinline__ float3 colliderProject(const PiesB200Collider& c, float3 x) {
  float3 n;
  const float phi = fminf(colliderPhi(c, x.x, x.y, x.z, &n), 0.0f);
  return make_float3(x.x - phi * n.x, x.y - phi * n.y, x.z - phi * n.z);
}

}  // namespace pies
