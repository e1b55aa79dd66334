// pd_kernels.cu — Projective Dynamics local step, RHS assembly and the per-substep
// streaming kernels (reference Src/Solver.cpp:229-238, :264-349, :386-395;
// Src/Constraints.cpp; Src/ShapeMatchingConstraint.cpp).
//
// All kernels are HBM/latency bound (largest dense object is a 3x3), so the rules
// are: 16 B vector accesses, plane-wise (SoA of float4) element tables that a warp
// reads as contiguous 512 B, node gathers through L1/L2, no atomics (every
// contribution has its own slot; a CSR gather sums them in a fixed order, which
// makes the right-hand side run-to-run bit-stable).
#include "kernels.h"
#include "rhs.cuh"
#include "svd3.cuh"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- inertia / momentum estimate (Solver.cpp:229-238) ------------------------------------
__global__ void __launch_bounds__(kThreads) k_predict(uint32_t n, float4* __restrict__ q,
                                                      const float4* __restrict__ vel,
                                                      float4* __restrict__ msn, float h) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i];
  float4 v = ldStream(vel + i);
  p.x += h * v.x; p.y += h * v.y; p.z += h * v.z;
  q[i] = p;
  float h2 = h * h;
  stStream(msn + i, make_float4(p.x / p.w / h2, p.y / p.w / h2, p.z / p.w / h2, 0.0f));
}

int launchPredict(cudaStream_t s, uint32_t n, float4* q, const float4* vel, float4* msn, float h) {
  if (!n) return 0;
  k_predict<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, q, vel, msn, h);
  return 1;
}

// ---- fused tet strain + volume projection (Constraints.cpp:76-128, :205-255) -----------------
// One thread per tet: gather 4 nodes, F = P Qinv, one SVD shared by both constraints,
// contribution_i = (w_s Fhat_s + w_v Fhat_v) Qinv^T (columns for nodes 2..4; node 1 gets
// minus their sum, i.e. w A^T B p with A = [0; Qinv^T D], B = I).
// The projection of element i, shared by k_tet_elems and k_tet_rhs; node(id) returns the position of node id.
template <typename NodeFn>
__device__ __forceinline__ void tetContribs(const TetElems& e, uint32_t i, NodeFn node, float4 (&out)[4]) {
  uint4 id = ldStream(e.ids + i);
  float4 qa = ldStream(e.qa + i), qb = ldStream(e.qb + i), pc = ldStream(e.pc + i), pd = ldStream(e.pd + i);
  float qinv[9] = {qa.x, qa.y, qa.z, qa.w, qb.x, qb.y, qb.z, qb.w, pc.x};
  V3 x1 = v3(node(id.x)), x2 = v3(node(id.y)), x3 = v3(node(id.z)), x4 = v3(node(id.w));
  M3 F = deformationGradient(x1, x2, x3, x4, qinv);
  M3 U, V;
  float sg[3];
  if (e.rot) {  // warm start from the factors of the previous PD iteration (state, like the shape-matching quaternion)
    float4 qu = e.rot[2ull * i], qv = e.rot[2ull * i + 1];
    svd3Warm(F, qu, qv, U, sg, V);
    e.rot[2ull * i] = qu; e.rot[2ull * i + 1] = qv;
  } else {
    svd3(F, U, sg, V);
  }
  float wS = pc.y, wV = pd.x;
  float d[3] = {0.0f, 0.0f, 0.0f};
  if (wS != 0.0f) {
    float t[3];
    strainSigma(sg, det3(F), pc.z, pc.w, t);
    d[0] += wS * t[0]; d[1] += wS * t[1]; d[2] += wS * t[2];
  }
  if (wV != 0.0f) {
    float t[3];
    volumeSigma(sg, pd.y, pd.z, t);
    d[0] += wV * t[0]; d[1] += wV * t[1]; d[2] += wV * t[2];
  }
  M3 T = recompose(U, d, V);  // w_s Fhat_s + w_v Fhat_v (both share U, V)
  V3 c[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {  // c_{k+1} = T * (row k of Qinv)
    float r0 = qinv[k], r1 = qinv[3 + k], r2 = qinv[6 + k];
    c[k] = v3(T.m[0][0] * r0 + T.m[0][1] * r1 + T.m[0][2] * r2,
              T.m[1][0] * r0 + T.m[1][1] * r1 + T.m[1][2] * r2,
              T.m[2][0] * r0 + T.m[2][1] * r1 + T.m[2][2] * r2);
  }
  // Node 1's row of A^T: the reference stores A(r,0) = fl(-(d_r0 + d_r1 + d_r2)) (Constraints.cpp:162),
  // whose rounding also sits in the system matrix; use the same rounded coefficients so the
  // right-hand side stays consistent with S (otherwise a position-proportional ghost force remains).
  float a0[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) a0[r] = __fadd_rn(__fadd_rn(-qinv[3 * r], -qinv[3 * r + 1]), -qinv[3 * r + 2]);
  V3 c0 = v3(T.m[0][0] * a0[0] + T.m[0][1] * a0[1] + T.m[0][2] * a0[2],
             T.m[1][0] * a0[0] + T.m[1][1] * a0[1] + T.m[1][2] * a0[2],
             T.m[2][0] * a0[0] + T.m[2][1] * a0[1] + T.m[2][2] * a0[2]);
  out[0] = f4(c0, 0.0f); out[1] = f4(c[0], 0.0f); out[2] = f4(c[1], 0.0f); out[3] = f4(c[2], 0.0f);
}

// list: the elements to project (null = 0 .. n-1)
__global__ void __launch_bounds__(128) k_tet_elems(TetElems e, const uint32_t* __restrict__ list, uint32_t n,
                                                   const float4* __restrict__ q, float4* __restrict__ contrib) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint32_t i = list ? list[t] : t;
  float4 c[4];
  tetContribs(e, i, [&](uint32_t id) { return __ldg(q + id); }, c);
  float4* out = contrib + 4ull * i;
  out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

int launchTetElems(cudaStream_t s, const TetElems& e, const uint32_t* list, uint32_t n, const float4* q, float4* contrib) {
  if (!n) return 0;
  k_tet_elems<<<gridFor(n, 128), 128, 0, s>>>(e, list, n, q, contrib);
  return 1;
}

// ---- fused local step + RHS over closed segments (HostSystem::segs) -------------------------------------
// One CTA per segment.  Its nodes' positions are staged in shared memory; each thread projects elements exactly like
// k_tet_elems and keeps their four contributions in shared memory; then each thread assembles nodes like
// k_gather_rhs_contacts: msn, plus the contributions in the order of the global gather list (slot = the same list in
// segment-local slots), plus the collision and floor terms.  The same code and the same sequence of float adds as the
// two-kernel path, so the same bits, without the contributions' round trip through HBM and the inc gather.
// Eight CTAs per SM (32 warps, 64 registers: a 52 B spill of loop state to L1) measured 75.0 us per iteration at S3 on a
// B200, seven (72 registers) 77.3 us, six (78, no spill) 81.3 us; one 256-thread CTA per segment 93.6 us.
// kColliders adds the static colliders' terms; the variant without them is launched whenever the solver has none.
template <bool kColliders>
__global__ void __launch_bounds__(kTetRhsThreads, 8) k_tet_rhs(TetElems e, TetSegments sg, const float4* __restrict__ q,
                                                            const float4* __restrict__ msn, const int* __restrict__ incPtr,
                                                            ContactLists c, const float4* __restrict__ contribC,
                                                            float4* __restrict__ snap, float4* __restrict__ rhs) {
  __shared__ float4 sQ[kSegNodes];
  __shared__ float4 sC[4 * kSegElems];
  const uint4 g = sg.segs[blockIdx.x];  // n0, n1, e0, e1
  const uint32_t nN = g.y - g.x, nE = g.w - g.z;
  for (uint32_t v = threadIdx.x; v < nN; v += kTetRhsThreads) sQ[v] = __ldg(q + g.x + v);
  __syncthreads();
  for (uint32_t t = threadIdx.x; t < nE; t += kTetRhsThreads) {
    float4 cv[4];
    tetContribs(e, g.z + t, [&](uint32_t id) { return sQ[id - g.x]; }, cv);
    sC[4 * t] = cv[0]; sC[4 * t + 1] = cv[1]; sC[4 * t + 2] = cv[2]; sC[4 * t + 3] = cv[3];
  }
  __syncthreads();
  for (uint32_t v = threadIdx.x; v < nN; v += kTetRhsThreads) {
    const uint32_t i = g.x + v;
    float4 acc = ldStream(msn + i);
    const int beg = incPtr[i], end = incPtr[i + 1];
    for (int k = beg; k < end; ++k) {
      const float4 cv = sC[sg.slot[k]];
      acc.x += cv.x; acc.y += cv.y; acc.z += cv.z;
    }
    addContactTerms<kColliders>(acc, i, c, contribC, q, snap);
    acc.w = 0.0f;
    rhs[i] = acc;
  }
}

int launchTetRhs(cudaStream_t s, const TetElems& e, const TetSegments& sg, const float4* q, const float4* msn,
                 const int* incPtr, const ContactLists& c, const float4* contribC, float4* snap, float4* rhs) {
  if (!sg.n) return 0;
  if (c.nCollide) k_tet_rhs<true><<<sg.n, kTetRhsThreads, 0, s>>>(e, sg, q, msn, incPtr, c, contribC, snap, rhs);
  else k_tet_rhs<false><<<sg.n, kTetRhsThreads, 0, s>>>(e, sg, q, msn, incPtr, c, contribC, snap, rhs);
  return 1;
}

// ---- distance (Constraints.cpp:11-37; A = B = 1/2 [1 -1; -1 1]) ------------------------------
__global__ void __launch_bounds__(kThreads) k_distance(DistanceElems e, const float4* __restrict__ q,
                                                       float4* __restrict__ contrib) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= e.n) return;
  uint2 id = e.ids[i];
  float2 rw = e.restW[i];
  V3 a = v3(__ldg(q + id.x)), b = v3(__ldg(q + id.y));
  V3 diff = b - a;
  float dist = length(diff);
  V3 dir = v3(1.0f, 0.0f, 0.0f);
  if (dist > 0.00001f) dir = diff / dist;
  float disp = rw.x - dist;
  V3 p0 = a + (-disp) * dir;
  V3 c0 = rw.y * (0.5f * p0 + (-0.5f) * b);
  V3 c1 = rw.y * ((-0.5f) * p0 + 0.5f * b);
  contrib[2ull * i] = f4(c0, 0.0f);
  contrib[2ull * i + 1] = f4(c1, 0.0f);
}

int launchDistance(cudaStream_t s, const DistanceElems& e, const float4* q, float4* contrib) {
  if (!e.n) return 0;
  k_distance<<<gridFor(e.n, kThreads), kThreads, 0, s>>>(e, q, contrib);
  return 1;
}

// ---- bend (Constraints.cpp:312-366; A = B = I4) ------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_bend(BendElems e, const float4* __restrict__ q,
                                                   float4* __restrict__ contrib) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= e.n) return;
  uint4 id = e.ids[i];
  float2 aw = e.angleW[i];
  float4 n1_ = __ldg(q + id.x), n2_ = __ldg(q + id.y), n3_ = __ldg(q + id.z), n4_ = __ldg(q + id.w);
  V3 x1 = v3(n1_), x2 = v3(n2_), x3 = v3(n3_), x4 = v3(n4_);
  V3 p2 = x2 - x1, p3 = x3 - x1, p4 = x4 - x1;
  V3 p2Xp3 = cross(p2, p3), p2Xp4 = cross(p2, p4);
  float l23 = length(p2Xp3), l24 = length(p2Xp4);
  V3 n1 = p2Xp3 / l23, n2 = p2Xp4 / l24;
  float d = dot(n1, n2);
  float C = (float)(acos((double)d) - (double)aw.x);  // the reference's unqualified acos() is the double overload
  V3 q3 = (cross(p2, n2) + cross(n1, p2) * d) / l23;
  V3 q4 = (cross(p2, n1) + cross(n2, p2) * d) / l24;
  V3 q2 = -((cross(p3, n2) + cross(n1, p3) * d) / l23) - ((cross(p4, n1) + cross(n2, p4) * d) / l24);
  V3 q1 = -q2 - q3 - q4;
  float wSum = n1_.w + n2_.w + n3_.w + n4_.w;
  float qq = dot(q1, q1) + dot(q2, q2) + dot(q3, q3) + dot(q4, q4);
  float om = 1.0f - d * d;
  float num = (float)(sqrt((double)(om < 0.0f ? 0.0f : om)) * (double)C);
  V3 o1 = x1, o2 = x2, o3 = x3, o4 = x4;
  if (!(qq < 0.00001f)) {
    o1 += -q1 * (4.0f * n1_.w / wSum) * num / qq;
    o2 += -q2 * (4.0f * n2_.w / wSum) * num / qq;
    o3 += -q3 * (4.0f * n3_.w / wSum) * num / qq;
    o4 += -q4 * (4.0f * n4_.w / wSum) * num / qq;
  }
  float4* out = contrib + 4ull * i;
  out[0] = f4(aw.y * o1, 0.0f); out[1] = f4(aw.y * o2, 0.0f);
  out[2] = f4(aw.y * o3, 0.0f); out[3] = f4(aw.y * o4, 0.0f);
}

int launchBend(cudaStream_t s, const BendElems& e, const float4* q, float4* contrib) {
  if (!e.n) return 0;
  k_bend<<<gridFor(e.n, kThreads), kThreads, 0, s>>>(e, q, contrib);
  return 1;
}

// ---- goal matching (ShapeMatchingConstraint.cpp:162-173): p = T (m, 1) -----------------------------
__global__ void __launch_bounds__(kThreads) k_goal(ClusterElems c, const float* __restrict__ material,
                                                   const float* __restrict__ xform, const float* __restrict__ w,
                                                   float4* __restrict__ contrib) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= c.nMembers) return;
  // cluster of member i: binary search in the offsets (clusters are few and cached)
  uint32_t lo = 0, hi = c.nClusters;
  while (hi - lo > 1) { uint32_t mid = (lo + hi) >> 1; if (c.off[mid] <= i) lo = mid; else hi = mid; }
  const float* T = xform + 16 * lo;
  float mx = material[3 * i], my = material[3 * i + 1], mz = material[3 * i + 2];
  float px = (T[0] * mx + T[4] * my) + (T[8] * mz + T[12]);
  float py = (T[1] * mx + T[5] * my) + (T[9] * mz + T[13]);
  float pz = (T[2] * mx + T[6] * my) + (T[10] * mz + T[14]);
  float ww = w[lo];
  contrib[i] = make_float4(ww * px, ww * py, ww * pz, 0.0f);
}

int launchGoal(cudaStream_t s, const ClusterElems& c, const float* material, const float* xform, const float* w,
               float4* contrib) {
  if (!c.nMembers) return 0;
  k_goal<<<gridFor(c.nMembers, kThreads), kThreads, 0, s>>>(c, material, xform, w, contrib);
  return 1;
}

// ---- shape matching (ShapeMatchingConstraint.cpp:75-122) --------------------------------------------
// One warp per cluster: lanes stride the members for the fp32 centroid and the fp64
// mass-weighted covariance, butterfly-reduce, then every lane runs the (cheap, uniform)
// warm-started rotation extraction in fp64 and projects its members.
__device__ __forceinline__ double warpSumD(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void quatToMatrix(const double (&q)[4] /*x y z w*/, double (&R)[3][3]) {
  double tx = 2.0 * q[0], ty = 2.0 * q[1], tz = 2.0 * q[2];
  double twx = tx * q[3], twy = ty * q[3], twz = tz * q[3];
  double txx = tx * q[0], txy = ty * q[0], txz = tz * q[0];
  double tyy = ty * q[1], tyz = tz * q[1], tzz = tz * q[2];
  R[0][0] = 1.0 - (tyy + tzz); R[0][1] = txy - twz; R[0][2] = txz + twy;
  R[1][0] = txy + twz; R[1][1] = 1.0 - (txx + tzz); R[1][2] = tyz - twx;
  R[2][0] = txz - twy; R[2][1] = tyz + twx; R[2][2] = 1.0 - (txx + tyy);
}

__global__ void __launch_bounds__(128) k_shape(ClusterElems c, const double* __restrict__ material,
                                               const double* __restrict__ qinv, double* __restrict__ quat,
                                               const float* __restrict__ w, const float4* __restrict__ q,
                                               float4* __restrict__ contrib) {
  uint32_t cluster = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (cluster >= c.nClusters) return;
  uint32_t beg = c.off[cluster], end = c.off[cluster + 1];
  uint32_t n = end - beg;
  if (n == 0) return;  // empty clusters exist (createShapeMatchingSheet quirk) and do nothing
  float weight = 1.0f / (float)n;
  float cx = 0.0f, cy = 0.0f, cz = 0.0f;
  for (uint32_t m = beg + lane; m < end; m += 32) {
    float4 p = __ldg(q + c.ids[m]);
    cx += weight * p.x; cy += weight * p.y; cz += weight * p.z;
  }
  cx = warpSum(cx); cy = warpSum(cy); cz = warpSum(cz);
  double P[3][3] = {{0, 0, 0}, {0, 0, 0}, {0, 0, 0}};
  for (uint32_t m = beg + lane; m < end; m += 32) {
    float4 p = __ldg(q + c.ids[m]);
    double l[3] = {(double)(p.x - cx), (double)(p.y - cy), (double)(p.z - cz)};
    double im = (double)p.w;
    const double* mc = material + 3ull * m;
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
      for (int cc = 0; cc < 3; ++cc) P[r][cc] += l[r] * mc[cc] / im;
  }
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) P[r][cc] = warpSumD(P[r][cc]);
  const double* Qi = qinv + 9ull * cluster;  // column-major
  double F[3][3];
#pragma unroll
  for (int r = 0; r < 3; ++r)
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) F[r][cc] = P[r][0] * Qi[3 * cc] + P[r][1] * Qi[3 * cc + 1] + P[r][2] * Qi[3 * cc + 2];
  double qt[4] = {quat[4ull * cluster], quat[4ull * cluster + 1], quat[4ull * cluster + 2], quat[4ull * cluster + 3]};
  double R[3][3];
  for (int iter = 0; iter < 100; ++iter) {  // Mueller et al., warm-started (stateful, SURVEY F11)
    quatToMatrix(qt, R);
    double ox = 0, oy = 0, oz = 0, dsum = 0;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      double rx = R[0][k], ry = R[1][k], rz = R[2][k], ax = F[0][k], ay = F[1][k], az = F[2][k];
      ox += ry * az - rz * ay; oy += rz * ax - rx * az; oz += rx * ay - ry * ax;
      dsum += rx * ax + ry * ay + rz * az;
    }
    double scale = 1.0 / fabs(dsum) + 1.0e-9;
    ox *= scale; oy *= scale; oz *= scale;
    double wn = sqrt(ox * ox + oy * oy + oz * oz);
    if (wn < 1.0e-9) break;
    double inv = 1.0 / wn;
    double sh, ch;
    sincos(0.5 * wn, &sh, &ch);
    double ax = sh * (inv * ox), ay = sh * (inv * oy), az = sh * (inv * oz), aw = ch;
    // q <- a * q
    double nx = aw * qt[0] + ax * qt[3] + ay * qt[2] - az * qt[1];
    double ny = aw * qt[1] + ay * qt[3] + az * qt[0] - ax * qt[2];
    double nz = aw * qt[2] + az * qt[3] + ax * qt[1] - ay * qt[0];
    double nw = aw * qt[3] - ax * qt[0] - ay * qt[1] - az * qt[2];
    double nn = 1.0 / sqrt(nx * nx + ny * ny + nz * nz + nw * nw);
    qt[0] = nx * nn; qt[1] = ny * nn; qt[2] = nz * nn; qt[3] = nw * nn;
  }
  if (lane == 0) {
    quat[4ull * cluster] = qt[0]; quat[4ull * cluster + 1] = qt[1];
    quat[4ull * cluster + 2] = qt[2]; quat[4ull * cluster + 3] = qt[3];
  }
  quatToMatrix(qt, R);
  double ww = (double)w[cluster];
  for (uint32_t m = beg + lane; m < end; m += 32) {
    const double* mc = material + 3ull * m;
    double px = R[0][0] * mc[0] + R[0][1] * mc[1] + R[0][2] * mc[2] + (double)cx;
    double py = R[1][0] * mc[0] + R[1][1] * mc[1] + R[1][2] * mc[2] + (double)cy;
    double pz = R[2][0] * mc[0] + R[2][1] * mc[1] + R[2][2] * mc[2] + (double)cz;
    contrib[m] = make_float4((float)(ww * px), (float)(ww * py), (float)(ww * pz), 0.0f);
  }
}

int launchShape(cudaStream_t s, const ClusterElems& c, const double* material, const double* qinv, double* quat,
                const float* w, const float4* q, float4* contrib) {
  if (!c.nClusters) return 0;
  k_shape<<<gridFor((uint64_t)c.nClusters * 32, 128), 128, 0, s>>>(c, material, qinv, quat, w, q, contrib);
  return 1;
}

// ---- RHS assembly: deterministic CSR gather (replaces Constraints.h:89-105 scatter-adds) ------------
// rhs_i = Msn_h2_i + sum over the node's incidences, in the reference's type order
// (position, distance, tet/volume, bend, shape, goal) then creation order.  nodes: the nodes to assemble (null = 0 .. n-1).
__global__ void __launch_bounds__(kThreads) k_gather_rhs(uint32_t n, const uint32_t* __restrict__ nodes,
                                                         const float4* __restrict__ msn,
                                                         const int* __restrict__ incPtr,
                                                         const uint32_t* __restrict__ inc,
                                                         const float4* __restrict__ contrib,
                                                         float4* __restrict__ rhs) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  const uint32_t i = nodes ? nodes[t] : t;
  float4 acc = ldStream(msn + i);
  int beg = incPtr[i], end = incPtr[i + 1];
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
  acc.w = 0.0f;
  rhs[i] = acc;
}

int launchGatherRhs(cudaStream_t s, uint32_t n, const uint32_t* nodes, const float4* msn, const int* incPtr,
                    const uint32_t* inc, const float4* contrib, float4* rhs) {
  if (!n) return 0;
  k_gather_rhs<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, nodes, msn, incPtr, inc, contrib, rhs);
  return 1;
}

// ---- velocity update (Solver.cpp:386-395) -----------------------------------------------------
// kForce adds the external force (forces.cu) as a final addition, (h f) invMass, rounded on its own; the variant without
// it is the reference's update and runs whenever the solver has no external force.
template <bool kForce>
__global__ void __launch_bounds__(kThreads) k_velocity(uint32_t n, const float4* __restrict__ q,
                                                       float4* __restrict__ prev, float4* __restrict__ vel,
                                                       float h, float damping, float gravity,
                                                       const float4* __restrict__ fext) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i];
  float4 pp = prev[i];
  float k = 1.0f - damping;
  float fy = -gravity / p.w;  // node.force = (0,-g,0)/invMass (Solver.cpp:224-226)
  float4 v;
  v.x = k * (p.x - pp.x) / h + h * 0.0f * p.w;
  v.y = k * (p.y - pp.y) / h + h * fy * p.w;
  v.z = k * (p.z - pp.z) / h + h * 0.0f * p.w;
  if constexpr (kForce) {
    const float4 f = ldStream(fext + i);
    v.x = __fadd_rn(v.x, __fmul_rn(__fmul_rn(h, f.x), p.w));
    v.y = __fadd_rn(v.y, __fmul_rn(__fmul_rn(h, f.y), p.w));
    v.z = __fadd_rn(v.z, __fmul_rn(__fmul_rn(h, f.z), p.w));
  }
  v.w = 0.0f;
  vel[i] = v;
  prev[i] = make_float4(p.x, p.y, p.z, pp.w);
}

int launchVelocityUpdate(cudaStream_t s, uint32_t n, const float4* q, float4* prev, float4* vel, float h,
                         float damping, float gravity, const float4* fext) {
  if (!n) return 0;
  if (fext) k_velocity<true><<<gridFor(n, kThreads), kThreads, 0, s>>>(n, q, prev, vel, h, damping, gravity, fext);
  else k_velocity<false><<<gridFor(n, kThreads), kThreads, 0, s>>>(n, q, prev, vel, h, damping, gravity, nullptr);
  return 1;
}

}  // namespace pies
