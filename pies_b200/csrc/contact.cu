// contact.cu — collision response of the PD path: per-iteration projections of the
// point-triangle / floor constraints, collision stabilisation and the friction pass.
//
// Reference: Src/CollisionConstraint.cpp:86-194 (point-triangle), :439-463 (floor),
// Src/Solver.cpp:298-308,337-349 (local step / RHS), :367-383 (stabilisation), :431-484 (friction).
//
// Stabilisation and friction are sequential Gauss-Seidel sweeps over the collision list in the
// reference, and the result depends on that order (SURVEY F8).  They run here as dataflow sweeps
// that honour exactly that order per node (k_gs_dataflow below).
#include "contact.h"
#include "reblock.h"

#include "common.cuh"
#include "rhs.cuh"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- per-iteration projections (parallel, no ordering issue) ---------------------------------------
// contribC[4u + slot] = copies * w * (A^T A p)_slot for distinct contact u, with p = current positions and
// p_A pushed to `thickness` above the triangle plane when below it (CollisionConstraint.cpp:86-124, :176-194).
// The reference adds the identical term once per copy; the copies are folded into the weight here.
__global__ void __launch_bounds__(kThreads) k_pt_project(uint32_t nTri, const uint4* __restrict__ entries,
                                                         const float* __restrict__ weight,
                                                         const float4* __restrict__ q, float thickness,
                                                         float4* __restrict__ contribC) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nTri) return;
  uint4 id = entries[e];
  const float kPtW = weight[e];  // copies * PointTriangleCollisionConstraint::w
  V3 A = v3(q[id.x]), B = v3(q[id.y]), C = v3(q[id.z]), D = v3(q[id.w]);
  V3 nrm = normalize(cross(C - B, D - B));
  float nDotP = dot(nrm, A - B);
  V3 pA = A;
  if (nDotP < thickness) pA += (thickness - nDotP) * nrm;
  V3 c0 = 3.0f * pA + (-1.0f) * B + (-1.0f) * C + (-1.0f) * D;
  contribC[4ull * e + 0] = f4(kPtW * c0, 0.0f);
  contribC[4ull * e + 1] = f4(kPtW * ((-1.0f) * pA + B), 0.0f);
  contribC[4ull * e + 2] = f4(kPtW * ((-1.0f) * pA + C), 0.0f);
  contribC[4ull * e + 3] = f4(kPtW * ((-1.0f) * pA + D), 0.0f);
}

// (the floor contacts' projectedPosition — CollisionConstraint.cpp:447-455: the position with y < 0 -> 0, the same for
// every duplicate of a node — is computed and stored per node by k_gather_rhs_contacts)
int launchContactProject(cudaStream_t s, const ContactLists& c, const float4* q, float thickness, float4* contribC) {
  int L = 0;
  if (c.nUnique) { k_pt_project<<<gridFor(c.nUnique, kThreads), kThreads, 0, s>>>(c.nUnique, c.uTri, c.uW, q, thickness, contribC); ++L; }
  return L;
}

// The whole right-hand side in one pass when there are contacts: the constraint gather of k_gather_rhs (pd_kernels.cu),
// then rhs_i += sum of the collision contributions (list order) + per floor duplicate w * projectedPosition
// (Solver.cpp:337-349), in that order; the floor contacts' projectedPosition (the position with y < 0 -> 0) is written to
// `snap` for the stabilisation sweeps, then the static colliders' terms when kColliders.  nodes: the nodes to assemble
// (null = 0 .. n-1).
template <bool kColliders>
__global__ void __launch_bounds__(kThreads) k_gather_rhs_contacts(uint32_t n, const uint32_t* __restrict__ nodes,
                                                                  const float4* __restrict__ msn,
                                                                  const int* __restrict__ incPtr,
                                                                  const uint32_t* __restrict__ inc,
                                                                  const float4* __restrict__ contrib, ContactLists c,
                                                                  const float4* __restrict__ contribC,
                                                                  const float4* __restrict__ q, float4* __restrict__ snap,
                                                                  float4* __restrict__ rhs) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint32_t i = nodes ? nodes[t] : t;
  float4 acc = ldStream(msn + i);
  {
    const int beg = incPtr[i], end = incPtr[i + 1];
    int k = beg;
    for (; k + 4 <= end; k += 4) {   // four gathers in flight; summed in list order (the result does not depend on the batching)
      const uint32_t j0 = inc[k], j1 = inc[k + 1], j2 = inc[k + 2], j3 = inc[k + 3];
      const float4 v0 = __ldg(contrib + j0), v1 = __ldg(contrib + j1), v2 = __ldg(contrib + j2), v3 = __ldg(contrib + j3);
      acc.x += v0.x; acc.y += v0.y; acc.z += v0.z;
      acc.x += v1.x; acc.y += v1.y; acc.z += v1.z;
      acc.x += v2.x; acc.y += v2.y; acc.z += v2.z;
      acc.x += v3.x; acc.y += v3.y; acc.z += v3.z;
    }
    for (; k < end; ++k) {
      float4 cv = __ldg(contrib + inc[k]);
      acc.x += cv.x; acc.y += cv.y; acc.z += cv.z;
    }
  }
  addContactTerms<kColliders>(acc, i, c, contribC, q, snap);
  acc.w = 0.0f;
  rhs[i] = acc;
}

int launchGatherRhsContacts(cudaStream_t s, uint32_t n, const uint32_t* nodes, const float4* msn, const int* incPtr,
                            const uint32_t* inc, const float4* contrib, const ContactLists& c, const float4* contribC,
                            const float4* q, float4* snap, float4* rhs) {
  if (!n) return 0;
  if (c.nCollide)
    k_gather_rhs_contacts<true><<<gridFor(n, kThreads), kThreads, 0, s>>>(n, nodes, msn, incPtr, inc, contrib, c, contribC, q, snap, rhs);
  else
    k_gather_rhs_contacts<false><<<gridFor(n, kThreads), kThreads, 0, s>>>(n, nodes, msn, incPtr, inc, contrib, c, contribC, q, snap, rhs);
  return 1;
}

// ---- ordered Gauss-Seidel executor (dataflow) ---------------------------------------------------------
// The reference sweeps the collision list sequentially; entry e reads and writes its four nodes, so the
// only constraint a parallel schedule has to respect is, per node, the list order of the entries that
// touch it.  Detection gives every (entry, node) its ticket = number of earlier entries touching that
// node.  Warps take chunks of 32 consecutive entries from a global counter (so every chunk below the
// newest one is owned by a running warp); an entry executes as soon as nodeDone[v] == ticket for its
// four nodes, then publishes nodeDone[v] = ticket + 1.  The earliest unfinished entry is always
// runnable, so the sweep cannot stall, and the result equals the sequential sweep up to rounding of
// the identical operations (same operand values, same order per node).
// (A chunk-level variant that runs the 32 entries of a chunk from shared memory was measured and dropped: at
// chunk granularity the false dependencies serialise a percolated pile, 29 ms per sweep instead of 1.1 ms.)
constexpr int kGsThreads = 256;

struct StabilizeOp {
  float4* q;
  float4* prev;
  float thickness;
  // PointTriangleCollisionConstraint::stabilizeCollisions (CollisionConstraint.cpp:126-162)
  __device__ __forceinline__ void operator()(uint4 id) const {
    float4 a4 = __ldcg(q + id.x), b4 = __ldcg(q + id.y), c4 = __ldcg(q + id.z), d4 = __ldcg(q + id.w);
    V3 A = v3(a4), B = v3(b4), C = v3(c4), D = v3(d4);
    V3 nrm = normalize(cross(C - B, D - B));
    float nDotP = dot(nrm, A - B);
    if (!(nDotP < thickness)) return;
    V3 disp = (thickness - nDotP) * nrm;
    float wTri = b4.w + c4.w + d4.w;
    float wSum = a4.w + wTri;
    V3 da = disp * a4.w / wSum, dt = disp * wTri / wSum;
    float4 pa = __ldcg(prev + id.x), pb = __ldcg(prev + id.y), pc = __ldcg(prev + id.z), pd = __ldcg(prev + id.w);
    __stcg(q + id.x, f4(A + da, a4.w)); __stcg(q + id.y, f4(B - dt, b4.w));
    __stcg(q + id.z, f4(C - dt, c4.w)); __stcg(q + id.w, f4(D - dt, d4.w));
    __stcg(prev + id.x, f4(v3(pa) + da, pa.w)); __stcg(prev + id.y, f4(v3(pb) - dt, pb.w));
    __stcg(prev + id.z, f4(v3(pc) - dt, pc.w)); __stcg(prev + id.w, f4(v3(pd) - dt, pd.w));
  }
};

struct FrictionOp {
  const float4* q;
  float4* vel;
  float friction, staticThreshold;
  // point-triangle friction / restitution (Solver.cpp:431-471); positions are not modified by this pass
  __device__ __forceinline__ void operator()(uint4 id) const {
    float4 a4 = q[id.x], b4 = q[id.y], c4 = q[id.z], d4 = q[id.w];
    V3 va = v3(__ldcg(vel + id.x)), vb = v3(__ldcg(vel + id.y)), vc = v3(__ldcg(vel + id.z)), vd = v3(__ldcg(vel + id.w));
    V3 avgTri = (vb + vc + vd) / 3.0f;
    V3 nrm = normalize(cross(v3(c4) - v3(b4), v3(d4) - v3(b4)));
    V3 rel = va - avgTri;
    float vDotN = dot(rel, nrm);
    V3 perp = rel - vDotN * nrm;
    float fr = friction;
    if (length(perp) < staticThreshold) fr = 1.0f;
    float triW = b4.w + c4.w + d4.w;
    float wSum = a4.w + triW;
    V3 dv = (-fr) * perp - (1.1f * fminf(vDotN, 0.0f)) * nrm;
    V3 dtv = (-dv) * triW / wSum;
    __stcg(vel + id.x, f4(va + dv * a4.w / wSum, 0.0f));
    __stcg(vel + id.y, f4(vb + dtv, 0.0f)); __stcg(vel + id.z, f4(vc + dtv, 0.0f)); __stcg(vel + id.w, f4(vd + dtv, 0.0f));
  }
};

template <typename Op>
__global__ void __launch_bounds__(kGsThreads) k_gs_dataflow(const uint4* __restrict__ entries,
                                                            const uint4* __restrict__ ticket, uint32_t nTri,
                                                            const uint8_t* __restrict__ gsClass,
                                                            uint32_t* __restrict__ nodeDone,
                                                            uint32_t* __restrict__ chunkCounter, Op op) {
  const int lane = threadIdx.x & 31;
  const uint32_t nChunks = (nTri + 31u) >> 5;
  while (true) {
    uint32_t chunk = 0;
    if (lane == 0) chunk = atomicAdd(chunkCounter, 1u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    if (chunk >= nChunks) break;
    uint32_t e = (chunk << 5) + (uint32_t)lane;
    bool pending = e < nTri;
    uint4 id = make_uint4(0, 0, 0, 0), tk = make_uint4(0, 0, 0, 0);
    if (pending) {
      id = entries[e];
      // entries of small clusters are swept inside one warp (k_gs_cluster_*); they share no node with the rest
      if (gsClass[id.x] != 2) pending = false; else tk = ticket[e];
    }
    while (__any_sync(0xffffffffu, pending)) {
      if (pending) {
        bool ready = ldAcquire(nodeDone + id.x) == tk.x && ldAcquire(nodeDone + id.y) == tk.y &&
                     ldAcquire(nodeDone + id.z) == tk.z && ldAcquire(nodeDone + id.w) == tk.w;
        if (ready) {
          op(id);
          __threadfence();
          stRelease(nodeDone + id.x, tk.x + 1u); stRelease(nodeDone + id.y, tk.y + 1u);
          stRelease(nodeDone + id.z, tk.z + 1u); stRelease(nodeDone + id.w, tk.w + 1u);
          pending = false;
        }
      }
    }
  }
}

// ---- ordered sweeps of small contact clusters inside one warp -------------------------------------------
// A contact cluster (connected component of the contact graph, reblock.cu) of <= 32 nodes never interacts
// with anything outside it during the sweeps, so one warp keeps its nodes in registers (lane = node),
// walks the cluster's entries in list order and exchanges operands with shuffles: the sequential order of
// the reference at register latency, all four stabilisation sweeps in one launch.
// Sorted-entry records: the sort only looks at the low kClusterBits of the key, so the rest travels as payload:
//   key = (rank a | rank b << 10 | rank c << 20 | rank d << 30) << kClusterBits | cluster,   value = list index
// (rank = position of the node inside its cluster; 10 bits cover the clusters the in-warp / in-CTA executors take,
// larger clusters never read them).
constexpr int kClusterBits = 24;

__global__ void __launch_bounds__(kThreads) k_entry_keys(uint32_t nTri, const uint4* __restrict__ entries,
                                                         const uint32_t* __restrict__ clusterOf,
                                                         const uint32_t* __restrict__ rankOf, uint64_t* __restrict__ keys,
                                                         uint32_t* __restrict__ entryOf, uint32_t* __restrict__ entCount) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nTri) return;
  uint4 id = entries[e];
  uint32_t c = clusterOf[id.x];
  uint64_t ranks = (uint64_t)(rankOf[id.x] & 1023u) | ((uint64_t)(rankOf[id.y] & 1023u) << 10) |
                   ((uint64_t)(rankOf[id.z] & 1023u) << 20) | ((uint64_t)(rankOf[id.w] & 1023u) << 30);
  keys[e] = (ranks << kClusterBits) | c;
  entryOf[e] = e;
  atomicAdd(entCount + c, 1u);
}

__device__ __forceinline__ V3 shflV3(float4 v, int src) {
  return v3(__shfl_sync(0xffffffffu, v.x, src), __shfl_sync(0xffffffffu, v.y, src), __shfl_sync(0xffffffffu, v.z, src));
}

__global__ void __launch_bounds__(kThreads) k_gs_cluster_stabilize(ClusterView cv, float4* __restrict__ q,
                                                                   float4* __restrict__ prev, const float4* __restrict__ snap,
                                                                   const uint32_t* __restrict__ floorMult, int haveFloor,
                                                                   float thickness, uint32_t sweeps) {
  const int lane = threadIdx.x & 31;
  const uint32_t warpsPerGrid = (gridDim.x * blockDim.x) >> 5;
  const uint32_t nC = *cv.nClusters;
  for (uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < nC; c += warpsPerGrid) {
    const uint32_t nb = cv.start[c], size = cv.start[c + 1] - nb;
    if (size > 32u) continue;  // large cluster: dataflow sweeps
    const bool have = (uint32_t)lane < size;
    const uint32_t node = have ? cv.nodes[nb + lane] : 0u;
    float4 q4 = make_float4(0.0f, 0.0f, 0.0f, 1.0f), p4 = q4, s4 = q4;
    bool onFloor = false;
    if (have) {
      q4 = q[node]; p4 = prev[node];
      onFloor = haveFloor && floorMult[node] != 0u;
      if (onFloor) s4 = snap[node];
    }
    const uint32_t eb = cv.entStart[c], ee = cv.entStart[c + 1];
    for (uint32_t sweep = 0; sweep < sweeps; ++sweep) {
      for (uint32_t base = eb; base < ee; base += 32) {
        const uint64_t myK = base + lane < ee ? cv.keys[base + lane] >> kClusterBits : 0ull;
        const uint32_t myW = (uint32_t)(myK & 31u) | ((uint32_t)(myK >> 10) & 31u) << 8 | ((uint32_t)(myK >> 20) & 31u) << 16 |
                             ((uint32_t)(myK >> 30) & 31u) << 24;
        const int cnt = (int)min(32u, ee - base);
        for (int i = 0; i < cnt; ++i) {
          const uint32_t lw = __shfl_sync(0xffffffffu, myW, i);
          const int la = lw & 31u, lb = (lw >> 8) & 31u, lc = (lw >> 16) & 31u, ld = (lw >> 24) & 31u;
          // PointTriangleCollisionConstraint::stabilizeCollisions (CollisionConstraint.cpp:126-162), as StabilizeOp
          V3 A = shflV3(q4, la), B = shflV3(q4, lb), C = shflV3(q4, lc), D = shflV3(q4, ld);
          float wa = __shfl_sync(0xffffffffu, q4.w, la), wb = __shfl_sync(0xffffffffu, q4.w, lb),
                wc = __shfl_sync(0xffffffffu, q4.w, lc), wd = __shfl_sync(0xffffffffu, q4.w, ld);
          V3 nrm = normalize(cross(C - B, D - B));
          float nDotP = dot(nrm, A - B);
          if (!(nDotP < thickness)) continue;
          V3 disp = (thickness - nDotP) * nrm;
          float wTri = wb + wc + wd;
          float wSum = wa + wTri;
          V3 da = disp * wa / wSum, dt = disp * wTri / wSum;
          if (lane == la) {
            q4.x += da.x; q4.y += da.y; q4.z += da.z; p4.x += da.x; p4.y += da.y; p4.z += da.z;
          } else if (lane == lb || lane == lc || lane == ld) {
            q4.x -= dt.x; q4.y -= dt.y; q4.z -= dt.z; p4.x -= dt.x; p4.y -= dt.y; p4.z -= dt.z;
          }
        }
      }
      if (onFloor) { q4.x = s4.x; q4.y = s4.y; q4.z = s4.z; }  // Solver.cpp:379-382, after the sweep's tri entries
    }
    if (have) { q[node] = q4; prev[node] = p4; }
  }
}

__global__ void __launch_bounds__(kThreads) k_gs_cluster_friction(ClusterView cv, const float4* __restrict__ q,
                                                                  float4* __restrict__ vel, float friction,
                                                                  float staticThreshold) {
  const int lane = threadIdx.x & 31;
  const uint32_t warpsPerGrid = (gridDim.x * blockDim.x) >> 5;
  const uint32_t nC = *cv.nClusters;
  for (uint32_t c = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; c < nC; c += warpsPerGrid) {
    const uint32_t nb = cv.start[c], size = cv.start[c + 1] - nb;
    if (size > 32u) continue;
    const bool have = (uint32_t)lane < size;
    const uint32_t node = have ? cv.nodes[nb + lane] : 0u;
    float4 q4 = make_float4(0.0f, 0.0f, 0.0f, 1.0f), v4 = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (have) { q4 = q[node]; v4 = vel[node]; }
    const uint32_t eb = cv.entStart[c], ee = cv.entStart[c + 1];
    for (uint32_t base = eb; base < ee; base += 32) {
      const uint64_t myK = base + lane < ee ? cv.keys[base + lane] >> kClusterBits : 0ull;
      const uint32_t myW = (uint32_t)(myK & 31u) | ((uint32_t)(myK >> 10) & 31u) << 8 | ((uint32_t)(myK >> 20) & 31u) << 16 |
                           ((uint32_t)(myK >> 30) & 31u) << 24;
      const int cnt = (int)min(32u, ee - base);
      for (int i = 0; i < cnt; ++i) {
        const uint32_t lw = __shfl_sync(0xffffffffu, myW, i);
        const int la = lw & 31u, lb = (lw >> 8) & 31u, lc = (lw >> 16) & 31u, ld = (lw >> 24) & 31u;
        // point-triangle friction / restitution (Solver.cpp:431-471), as FrictionOp
        V3 B = shflV3(q4, lb), C = shflV3(q4, lc), D = shflV3(q4, ld);
        float wa = __shfl_sync(0xffffffffu, q4.w, la), wb = __shfl_sync(0xffffffffu, q4.w, lb),
              wc = __shfl_sync(0xffffffffu, q4.w, lc), wd = __shfl_sync(0xffffffffu, q4.w, ld);
        V3 va = shflV3(v4, la), vb = shflV3(v4, lb), vc = shflV3(v4, lc), vd = shflV3(v4, ld);
        V3 avgTri = (vb + vc + vd) / 3.0f;
        V3 nrm = normalize(cross(C - B, D - B));
        V3 rel = va - avgTri;
        float vDotN = dot(rel, nrm);
        V3 perp = rel - vDotN * nrm;
        float fr = friction;
        if (length(perp) < staticThreshold) fr = 1.0f;
        float triW = wb + wc + wd;
        float wSum = wa + triW;
        V3 dv = (-fr) * perp - (1.1f * fminf(vDotN, 0.0f)) * nrm;
        V3 dtv = (-dv) * triW / wSum;
        if (lane == la) {
          V3 nv = va + dv * wa / wSum;
          v4.x = nv.x; v4.y = nv.y; v4.z = nv.z;
        } else if (lane == lb || lane == lc || lane == ld) {
          v4.x += dtv.x; v4.y += dtv.y; v4.z += dtv.z;
        }
      }
    }
    if (have) vel[node] = make_float4(v4.x, v4.y, v4.z, 0.0f);
  }
}

// ---- ordered sweeps of mid-size contact clusters: one CTA, nodes staged in shared memory ----------------------
// A cluster of 33 .. kMidClusterMax nodes (a column of stacked bodies, a small pile) chains its entries through
// shared nodes, and the global dataflow executor pays an L2 round trip per link of that chain.  Here one CTA
// copies the cluster's nodes into shared memory and runs the same ticketed dataflow there: warps take chunks of 32
// consecutive entries (list order) from a shared counter, an entry runs once sDone[v] == ticket for its four nodes
// and publishes ticket + 1.  All sweeps and their floor snaps happen in one launch.  Clusters are independent, so
// which CTA takes which cluster does not matter; per node the order is the reference's sequential order.
constexpr int kMidThreads = 256;
constexpr int kMidCtasPerSm = 4;

__device__ __forceinline__ float4 ldsVolatile(const float4* p) {
  float4 v;
  asm volatile("ld.volatile.shared.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
  return v;
}
__device__ __forceinline__ void stsVolatile(float4* p, float4 v) {
  asm volatile("st.volatile.shared.v4.f32 [%0], {%1, %2, %3, %4};"
               ::"r"((uint32_t)__cvta_generic_to_shared(p)), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ uint32_t ldsVolatile(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"((uint32_t)__cvta_generic_to_shared(p)) : "memory");
  return v;
}
__device__ __forceinline__ void stsVolatile(uint32_t* p, uint32_t v) {
  asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(p)), "r"(v) : "memory");
}

// kStabilize: s0 = position, s1 = prevPosition, `sweeps` sweeps with the floor snap after each (StabilizeOp);
// otherwise s0 = position (read only), s1 = velocity, one sweep (FrictionOp).
template <bool kStabilize>
__global__ void __launch_bounds__(kMidThreads, kMidCtasPerSm) k_gs_mid(ClusterView cv, const uint32_t* __restrict__ nMidPtr,
                                                                      const uint4* __restrict__ ticket,
                                                                      float4* __restrict__ g0, float4* __restrict__ g1,
                                                                      const float4* __restrict__ snap,
                                                                      const uint32_t* __restrict__ floorMult, int haveFloor,
                                                                      float pa /* thickness | friction */,
                                                                      float pb /* - | staticThreshold */, uint32_t sweeps) {
  __shared__ float4 s0[kMidClusterMax], s1[kMidClusterMax];
  __shared__ uint32_t sDone[kMidClusterMax];
  __shared__ uint32_t sChunk;
  const int lane = threadIdx.x & 31;
  const uint32_t nMid = *nMidPtr;
  for (uint32_t mi = blockIdx.x; mi < nMid; mi += gridDim.x) {
    const uint32_t c = cv.midList[mi];
    const uint32_t nb = cv.start[c], size = cv.start[c + 1] - nb;
    for (uint32_t k = threadIdx.x; k < size; k += kMidThreads) {
      const uint32_t node = cv.nodes[nb + k];
      s0[k] = g0[node]; s1[k] = g1[node];
    }
    const uint32_t eb = cv.entStart[c], ee = cv.entStart[c + 1];
    const uint32_t nChunks = (ee - eb + 31u) >> 5;
    for (uint32_t sweep = 0; sweep < sweeps; ++sweep) {
      for (uint32_t k = threadIdx.x; k < size; k += kMidThreads) sDone[k] = 0u;
      if (threadIdx.x == 0) sChunk = 0u;
      __syncthreads();
      while (true) {
        uint32_t chunk = 0;
        if (lane == 0) chunk = atomicAdd(&sChunk, 1u);
        chunk = __shfl_sync(0xffffffffu, chunk, 0);
        if (chunk >= nChunks) break;
        const uint32_t pos = eb + (chunk << 5) + (uint32_t)lane;
        bool pending = pos < ee;
        uint32_t ra = 0, rb = 0, rc = 0, rd = 0;
        uint4 tk = make_uint4(0, 0, 0, 0);
        if (pending) {
          const uint64_t r = cv.keys[pos] >> kClusterBits;
          ra = (uint32_t)r & 1023u; rb = (uint32_t)(r >> 10) & 1023u; rc = (uint32_t)(r >> 20) & 1023u; rd = (uint32_t)(r >> 30) & 1023u;
          tk = ticket[cv.entryOf[pos]];
        }
        while (__any_sync(0xffffffffu, pending)) {
          if (pending) {
            const bool ready = ldsVolatile(sDone + ra) == tk.x && ldsVolatile(sDone + rb) == tk.y &&
                               ldsVolatile(sDone + rc) == tk.z && ldsVolatile(sDone + rd) == tk.w;
            if (ready) {
              __threadfence_block();
              const float4 a4 = ldsVolatile(s0 + ra), b4 = ldsVolatile(s0 + rb), c4 = ldsVolatile(s0 + rc), d4 = ldsVolatile(s0 + rd);
              if (kStabilize) {
                // PointTriangleCollisionConstraint::stabilizeCollisions (CollisionConstraint.cpp:126-162), as StabilizeOp
                V3 A = v3(a4), B = v3(b4), C = v3(c4), D = v3(d4);
                V3 nrm = normalize(cross(C - B, D - B));
                float nDotP = dot(nrm, A - B);
                if (nDotP < pa) {
                  V3 disp = (pa - nDotP) * nrm;
                  float wTri = b4.w + c4.w + d4.w;
                  float wSum = a4.w + wTri;
                  V3 da = disp * a4.w / wSum, dt = disp * wTri / wSum;
                  const float4 p0 = ldsVolatile(s1 + ra), p1 = ldsVolatile(s1 + rb), p2 = ldsVolatile(s1 + rc), p3 = ldsVolatile(s1 + rd);
                  stsVolatile(s0 + ra, f4(A + da, a4.w)); stsVolatile(s0 + rb, f4(B - dt, b4.w));
                  stsVolatile(s0 + rc, f4(C - dt, c4.w)); stsVolatile(s0 + rd, f4(D - dt, d4.w));
                  stsVolatile(s1 + ra, f4(v3(p0) + da, p0.w)); stsVolatile(s1 + rb, f4(v3(p1) - dt, p1.w));
                  stsVolatile(s1 + rc, f4(v3(p2) - dt, p2.w)); stsVolatile(s1 + rd, f4(v3(p3) - dt, p3.w));
                }
              } else {
                // point-triangle friction / restitution (Solver.cpp:431-471), as FrictionOp
                const V3 va = v3(ldsVolatile(s1 + ra)), vb = v3(ldsVolatile(s1 + rb)), vc = v3(ldsVolatile(s1 + rc)), vd = v3(ldsVolatile(s1 + rd));
                V3 avgTri = (vb + vc + vd) / 3.0f;
                V3 nrm = normalize(cross(v3(c4) - v3(b4), v3(d4) - v3(b4)));
                V3 rel = va - avgTri;
                float vDotN = dot(rel, nrm);
                V3 perp = rel - vDotN * nrm;
                float fr = pa;
                if (length(perp) < pb) fr = 1.0f;
                float triW = b4.w + c4.w + d4.w;
                float wSum = a4.w + triW;
                V3 dv = (-fr) * perp - (1.1f * fminf(vDotN, 0.0f)) * nrm;
                V3 dtv = (-dv) * triW / wSum;
                stsVolatile(s1 + ra, f4(va + dv * a4.w / wSum, 0.0f));
                stsVolatile(s1 + rb, f4(vb + dtv, 0.0f)); stsVolatile(s1 + rc, f4(vc + dtv, 0.0f)); stsVolatile(s1 + rd, f4(vd + dtv, 0.0f));
              }
              __threadfence_block();
              stsVolatile(sDone + ra, tk.x + 1u); stsVolatile(sDone + rb, tk.y + 1u);
              stsVolatile(sDone + rc, tk.z + 1u); stsVolatile(sDone + rd, tk.w + 1u);
              pending = false;
            }
          }
        }
      }
      __syncthreads();
      if (kStabilize && haveFloor) {  // Solver.cpp:379-382, after the sweep's point-triangle entries
        for (uint32_t k = threadIdx.x; k < size; k += kMidThreads) {
          const uint32_t node = cv.nodes[nb + k];
          if (floorMult[node] != 0u) { const float4 s4 = snap[node]; s0[k] = make_float4(s4.x, s4.y, s4.z, s0[k].w); }
        }
      }
      __syncthreads();
    }
    for (uint32_t k = threadIdx.x; k < size; k += kMidThreads) {
      const uint32_t node = cv.nodes[nb + k];
      if (kStabilize) { g0[node] = s0[k]; g1[node] = s1[k]; }
      else g1[node] = make_float4(s1[k].x, s1[k].y, s1[k].z, 0.0f);
    }
    __syncthreads();
  }
}

// nodes on the floor go back to their projected position (Solver.cpp:379-382)
__global__ void __launch_bounds__(kThreads) k_floor_snap(uint32_t nFloor, const uint32_t* __restrict__ nodes,
                                                         const float4* __restrict__ snap, float4* __restrict__ q,
                                                         const uint8_t* __restrict__ gsClass, int cls) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nFloor) return;
  uint32_t node = nodes[i];
  if (gsClass && gsClass[node] != cls) return;  // nodes of contact clusters are snapped inside their sweeps
  float4 p = snap[node];
  float4 cur = q[node];
  q[node] = make_float4(p.x, p.y, p.z, cur.w);
}

// floor friction, once per duplicate in list order (Solver.cpp:473-484); duplicates only touch their own node
__global__ void __launch_bounds__(kThreads) k_floor_friction(uint32_t n, const uint32_t* __restrict__ mult,
                                                             float4* __restrict__ vel, float friction, float staticThreshold) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t m = mult[i];
  if (!m) return;
  float4 v = vel[i];
  for (uint32_t k = 0; k < m; ++k) {
    float fr = friction;
    if (sqrtf(v.x * v.x + 0.0f + v.z * v.z) < staticThreshold) fr = 1.0f;
    v.x += (-fr) * v.x; v.y += (-fr) * 0.0f; v.z += (-fr) * v.z;
  }
  vel[i] = v;
}

constexpr int kSweepCounters = 64;

int prepareContactSweeps(ContactWork& w, cudaStream_t s, const ContactLists& c) {
  w.nTri = c.nTri;
  w.sweepsUsed = 0;
  w.haveClusters = false;
  if (!c.nTri) return 0;
  if (w.sweepCounters.reserve(kSweepCounters) != cudaSuccess) return -1;
  if (cudaMemsetAsync(w.sweepCounters.p, 0, kSweepCounters * sizeof(uint32_t), s) != cudaSuccess) return -1;
  return 0;
}

// After reblock.cu has formed this substep's contact clusters: entries grouped by cluster (stable, so list
// order survives inside a cluster) with the lanes of their four nodes.
int prepareClusterSweeps(ContactWork& w, cudaStream_t s, const ContactLists& c, const ClusterTables& t) {
  if (!c.nTri || !t.nTouched) return 0;
  const uint32_t nTri = c.nTri, clusterBound = t.nTouched / 4 + 2;
  if (w.keys.reserve(nTri) != cudaSuccess || w.tmpKeys.reserve(nTri) != cudaSuccess || w.lanes.reserve(nTri) != cudaSuccess ||
      w.tmpVals.reserve(nTri) != cudaSuccess || w.entStart.reserve(clusterBound + 2) != cudaSuccess ||
      w.sortHist.reserve(sortHistBytes(nTri) / 4 + 4) != cudaSuccess ||
      w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(clusterBound + 2, 1024))) != cudaSuccess)
    return -1;
  int L = 0;
  cudaMemsetAsync(w.entStart.p, 0, (size_t)(clusterBound + 2) * sizeof(uint32_t), s);
  k_entry_keys<<<gridFor(nTri, kThreads), kThreads, 0, s>>>(nTri, c.tri, t.clusterOf, t.rankOf, w.keys.p, w.lanes.p, w.entStart.p); ++L;
  L += launchExclusiveScan(s, w.entStart.p, clusterBound + 1, w.scanScratch.p);
  int bits = 1;
  while ((1ull << bits) <= (uint64_t)clusterBound) ++bits;
  if (bits > kClusterBits) return -1;  // > 16 M contact clusters in one substep: beyond the sorted-entry record layout
  L += launchSortPairs(s, nTri, w.keys.p, w.lanes.p, w.tmpKeys.p, w.tmpVals.p, w.sortHist.p, bits);
  w.view = ClusterView{t.nClusters, t.start, t.nodes, w.entStart.p, w.lanes.p, w.keys.p, t.midList};
  w.gsClass = t.gsClass;
  w.hostCounts = t.hostCounts; w.countsReady = t.countsReady; w.nMidDev = t.nMidDev;
  w.clusterBound = clusterBound;
  w.haveClusters = true;
  return L;
}

template <typename Op>
static int launchSweep(cudaStream_t s, ContactWork& w, const ContactLists& c, uint32_t n, Op op) {
  if (w.sweepsUsed == kSweepCounters) {  // more sweeps than counters in one substep: recycle
    cudaMemsetAsync(w.sweepCounters.p, 0, kSweepCounters * sizeof(uint32_t), s);
    w.sweepsUsed = 0;
  }
  cudaMemsetAsync(c.nodeDone, 0, (size_t)n * sizeof(uint32_t), s);
  uint32_t chunks = (c.nTri + 31u) / 32u;
  int grid = (int)std::min<uint32_t>(kNumSMs * 8, (chunks + kGsThreads / 32 - 1) / (kGsThreads / 32));
  k_gs_dataflow<Op><<<grid, kGsThreads, 0, s>>>(c.tri, c.ticket, c.nTri, w.gsClass, c.nodeDone,
                                                 w.sweepCounters.p + w.sweepsUsed, op);
  ++w.sweepsUsed;
  return 1;
}

static int clusterGrid(uint32_t clusterBound) {
  return (int)std::min<uint32_t>(kNumSMs * 8, (clusterBound + kThreads / 32 - 1) / (kThreads / 32));
}

// side stream + events of the concurrent mid-cluster sweeps, created at first use; false = run everything on s
static bool sideStream(ContactWork& w) {
  if (w.side) return true;
  if (cudaStreamCreateWithFlags(&w.side, cudaStreamNonBlocking) != cudaSuccess) { w.side = nullptr; cudaGetLastError(); return false; }
  if (cudaEventCreateWithFlags(&w.fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&w.join, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); return false; }
  return true;
}

int launchStabilize(cudaStream_t s, ContactWork& w, const ContactLists& c, uint32_t n, float4* q, float4* prev,
                    const float4* snap, float thickness, uint32_t iterations) {
  int L = 0;
  if (!iterations) return 0;
  const uint8_t* cls = (c.nTri && w.haveClusters) ? w.gsClass : nullptr;
  if (cls) {
    // how many mid / large clusters this substep has was copied to the host right after they were formed
    if (w.countsReady) cudaEventSynchronize(w.countsReady);
    const uint32_t nMid = w.hostCounts ? w.hostCounts[0] : 0u, nLarge = w.hostCounts ? w.hostCounts[1] : 1u;
    const bool aside = nMid && sideStream(w);
    if (aside) { cudaEventRecord(w.fork, s); cudaStreamWaitEvent(w.side, w.fork, 0); }
    if (nMid) {  // mid-size clusters: one CTA each, on the side stream, beside the small clusters below
      k_gs_mid<true><<<(int)std::min<uint32_t>(nMid, kNumSMs * kMidCtasPerSm), kMidThreads, 0, aside ? w.side : s>>>(
          w.view, w.nMidDev, c.ticket, q, prev, snap, c.floorMult, c.nFloor ? 1 : 0, thickness, 0.0f, iterations); ++L;
      if (aside) cudaEventRecord(w.join, w.side);
    }
    // small clusters: all sweeps (and their floor snaps) in one launch
    k_gs_cluster_stabilize<<<clusterGrid(w.clusterBound), kThreads, 0, s>>>(w.view, q, prev, snap, c.floorMult, c.nFloor ? 1 : 0,
                                                                           thickness, iterations); ++L;
    if (aside) cudaStreamWaitEvent(s, w.join, 0);
    // large clusters: dataflow sweeps, floor snap of their nodes after each one
    for (uint32_t it = 0; nLarge && it < iterations; ++it) {
      L += launchSweep(s, w, c, n, StabilizeOp{q, prev, thickness});
      if (c.nFloor) { k_floor_snap<<<gridFor(c.nFloor, kThreads), kThreads, 0, s>>>(c.nFloor, c.floorNode, snap, q, cls, 2); ++L; }
    }
  }
  // floor nodes outside every cluster: the snap is idempotent, once is the same as once per sweep
  if (c.nFloor) { k_floor_snap<<<gridFor(c.nFloor, kThreads), kThreads, 0, s>>>(c.nFloor, c.floorNode, snap, q, cls, 0); ++L; }
  return L;
}

int launchFriction(cudaStream_t s, ContactWork& w, const ContactLists& c, uint32_t n, const float4* q, float4* vel,
                   float friction, float staticThreshold) {
  int L = 0;
  if (c.nTri && w.haveClusters) {
    if (w.countsReady) cudaEventSynchronize(w.countsReady);
    const uint32_t nMid = w.hostCounts ? w.hostCounts[0] : 0u, nLarge = w.hostCounts ? w.hostCounts[1] : 1u;
    const bool aside = nMid && sideStream(w);
    if (aside) { cudaEventRecord(w.fork, s); cudaStreamWaitEvent(w.side, w.fork, 0); }
    if (nMid) {
      k_gs_mid<false><<<(int)std::min<uint32_t>(nMid, kNumSMs * kMidCtasPerSm), kMidThreads, 0, aside ? w.side : s>>>(
          w.view, w.nMidDev, c.ticket, const_cast<float4*>(q), vel, nullptr, nullptr, 0, friction, staticThreshold, 1u); ++L;
      if (aside) cudaEventRecord(w.join, w.side);
    }
    k_gs_cluster_friction<<<clusterGrid(w.clusterBound), kThreads, 0, s>>>(w.view, q, vel, friction, staticThreshold); ++L;
    if (aside) cudaStreamWaitEvent(s, w.join, 0);
    if (nLarge) L += launchSweep(s, w, c, n, FrictionOp{q, vel, friction, staticThreshold});
  }
  if (c.nFloor) { k_floor_friction<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, c.floorMult, vel, friction, staticThreshold); ++L; }
  return L;
}

// Loads this file's kernels now (CUDA loads a kernel lazily at its first launch; for the collision kernels that
// would be the first contact tick of a run, ~1 ms each in the middle of the simulation).
void preloadContactKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_pt_project);
  cudaFuncGetAttributes(&a, k_gs_dataflow<StabilizeOp>);
  cudaFuncGetAttributes(&a, k_gs_dataflow<FrictionOp>);
  cudaFuncGetAttributes(&a, k_entry_keys);
  cudaFuncGetAttributes(&a, k_gs_cluster_stabilize);
  cudaFuncGetAttributes(&a, k_gs_cluster_friction);
  cudaFuncGetAttributes(&a, k_gs_mid<true>);
  cudaFuncGetAttributes(&a, k_gs_mid<false>);
  cudaFuncGetAttributes(&a, k_floor_snap);
  cudaFuncGetAttributes(&a, k_gather_rhs_contacts<false>);
  cudaFuncGetAttributes(&a, k_gather_rhs_contacts<true>);
  cudaFuncGetAttributes(&a, k_floor_friction);
}

}  // namespace pies
