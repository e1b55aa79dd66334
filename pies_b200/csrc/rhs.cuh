// rhs.cuh — the collision and floor terms of the right-hand side (Solver.cpp:337-349), shared by the two kernels that
// assemble it with contacts: k_gather_rhs_contacts (contact.cu) and the fused local step k_tet_rhs (pd_kernels.cu).
// Both paths must produce the same bits, so these float adds exist once.
#pragma once

#include "common.cuh"
#include "kernels.h"

namespace pies {

constexpr float kFloorW = 10000.0f;  // StaticCollisionConstraint::w (CollisionConstraint.h:78)

// acc += the collision contributions of node i (list order), then w * projectedPosition once per floor duplicate; the
// floor contacts' projectedPosition (the position with y < 0 -> 0) is written to `snap` for the stabilisation sweeps.
// kColliders: then the static colliders' terms, c.colRhs[i] (formed by k_collider_project), for a node with a mask.
// A no-op when the substep has no contacts.
template <bool kColliders>
__device__ __forceinline__ void addContactTerms(float4& acc, uint32_t i, const ContactLists& c,
                                                const float4* __restrict__ contribC, const float4* __restrict__ q,
                                                float4* __restrict__ snap) {
  int beg = 0, end = 0;
  if (c.nTri) { beg = c.incPtr[i]; end = c.incPtr[i + 1]; }
  const uint32_t mult = c.nFloor ? c.floorMult[i] : 0u;
  for (int k = beg; k < end; ++k) {
    float4 v = contribC[c.inc[k]];
    acc.x += v.x; acc.y += v.y; acc.z += v.z;
  }
  if (mult) {
    float4 p = q[i];
    if (p.y < 0.0f) p.y = 0.0f;
    snap[i] = p;
    for (uint32_t k = 0; k < mult; ++k) { acc.x += kFloorW * p.x; acc.y += kFloorW * p.y; acc.z += kFloorW * p.z; }
  }
  if (kColliders && c.colMask[i]) {
    const float4 p = c.colRhs[i];
    acc.x += p.x; acc.y += p.y; acc.z += p.z;
  }
}

}  // namespace pies
