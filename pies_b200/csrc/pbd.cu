// pbd.cu — Position-Based-Dynamics time loop (reference Solver::tickPBD, Src/Solver.cpp:40-160).
//
// The reference is one sequential Gauss-Seidel: every projection reads positions the previous
// one wrote.  The parallel schedule here executes EXACTLY that order wherever two operations
// touch the same node and runs everything else concurrently:
//
//  * position / distance / bend constraints (Constraints.h:121-129 projectNodePositions) are swept
//    by a dataflow kernel: op k carries, for each node it touches, its ticket = number of earlier
//    ops touching that node (host-built once per topology); it runs when every node's progress
//    counter equals its ticket.  A chain created even-then-odd therefore runs as two colour
//    batches, a body lattice as its dependency levels, and independent bodies fully in parallel.
//  * the node hash (SpatialHash<Node>, NodeCompRange, Solver.cpp:81-82,877-901) is a radix sort of
//    (cell key, node) pairs + a cell-start table, rebuilt every iteration like the reference's.
//  * node-node response (Solver.cpp:85-130) visits, for node i in index order, every member j of every
//    bucket in i's range (range taken from i's position when its turn starts, buckets from the
//    positions at hash build).  Visits whose pair cannot overlap are no-ops in the reference (disp <= 0:
//    continue), so the visit list keeps only pairs within r_i + r_j + 2*delta at build time and cells
//    within delta of i's range, in the reference's (i, cell, j) order, and executes them as a
//    dataflow sweep.  delta bounds how far a node may move during the sweep; it is VERIFIED after the
//    sweep and the pass is redone from the saved positions with a larger delta if it was exceeded,
//    so the result never depends on the pruning.
//  * velocity edits inside the collision loop (Solver.cpp:113-125) are dead: the substep end
//    overwrites every velocity (Solver.cpp:143, SURVEY F4); they are not executed.
//
// Arithmetic uses the unfused round-to-nearest helpers of ccd.cuh in the reference's
// association order (the reference is built for baseline x86-64, no FMA).
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "ccd.cuh"
#include "engine.h"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

constexpr int kSweepThreads = 256;

struct PbdWork {
  uint64_t builtVersion = ~0ull;
  // constraint sweeps: ids / tickets per op (host-built), parameters
  DevBuf<uint32_t> posIds, posTk; DevBuf<float4> posTargetW;
  DevBuf<uint2> distIds, distTk; DevBuf<float2> distRestW;
  DevBuf<uint4> bendIds, bendTk; DevBuf<float2> bendAngleW;
  uint32_t nPos = 0, nDist = 0, nBend = 0;
  DevBuf<uint32_t> nodeDone, counters;   // progress counters; chunk counters of the sweeps
  uint32_t countersUsed = 0;
  // node hash
  DevBuf<int4> nodeMin; DevBuf<uint32_t> nodeLen, cnt, heads, cellStart, vals, tmpVals, sortHist, scanScratch;
  DevBuf<uint64_t> keys, tmpKeys, cellKey;
  DevBuf<int> bbox;
  DevBuf<float4> q0, turnStart;
  // visit list
  DevBuf<uint32_t> visCnt; DevBuf<uint4> visits /* i, j, keyLo, keyHi|first<<31 */; DevBuf<uint2> visTk;
  DevBuf<uint64_t> incKeys, incTmpKeys; DevBuf<uint32_t> incVals, incTmpVals, incPtr;
  DevBuf<uint32_t> flags;   // [0] movement bound exceeded
  // colour-batched node-node response (opt-in, PiesB200Tuning::reserved & 1024): distinct pairs, their colours
  DevBuf<uint32_t> pairCnt; DevBuf<uint4> pairs /* a, b, applications, - */; DevBuf<uint32_t> pairColor, nodeMinPrio;
  DevBuf<unsigned long long> nodeMask; DevBuf<uint32_t> colorStat;  // [0] pairs still uncoloured, [1] colours in use
  int* host = nullptr;      // pinned, 16 ints
  float delta = 0.0f;
  uint64_t visitsLastTick = 0;
  uint32_t nCells = 0; uint64_t nPairs = 0;
  int keyPack[5] = {0, 0, 0, 0, 0};
  cudaError_t lastError = cudaSuccess;
};

void destroyPbdWork(PbdWork* w) {
  if (!w) return;
  if (w->host) cudaFreeHost(w->host);
  delete w;
}

// ------------------------------------------------------------------------------------------
// streaming kernels
// advect (Solver.cpp:47-52): prev = pos; pos += v dt + (0,-g,0) dt dt
// kForce adds the external force (forces.cu) as a final addition, ((f invMass) dt) dt; the variant without it is the
// reference's advection and runs whenever the solver has no external force.
template <bool kForce>
__global__ void __launch_bounds__(kThreads) k_pbd_advect(uint32_t n, float4* __restrict__ q, float4* __restrict__ prev,
                                                         const float4* __restrict__ vel, float dt, float gravity,
                                                         const float4* __restrict__ fext) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i], o = prev[i], v = vel[i];
  prev[i] = make_float4(p.x, p.y, p.z, o.w);
  float gy = ex::mul(ex::mul(-gravity, dt), dt);
  p.x = ex::add(p.x, ex::add(ex::mul(v.x, dt), 0.0f));
  p.y = ex::add(p.y, ex::add(ex::mul(v.y, dt), gy));
  p.z = ex::add(p.z, ex::add(ex::mul(v.z, dt), 0.0f));
  if constexpr (kForce) {
    const float4 f = fext[i];
    p.x = ex::add(p.x, ex::mul(ex::mul(ex::mul(f.x, p.w), dt), dt));
    p.y = ex::add(p.y, ex::mul(ex::mul(ex::mul(f.y, p.w), dt), dt));
    p.z = ex::add(p.z, ex::mul(ex::mul(ex::mul(f.z, p.w), dt), dt));
  }
  q[i] = p;
}

// floor clamp (Solver.cpp:132-136)
__global__ void __launch_bounds__(kThreads) k_pbd_floor(uint32_t n, float4* __restrict__ q, const float4* __restrict__ prev,
                                                        float floorHeight) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i];
  float r = prev[i].w;
  if (ex::sub(p.y, r) < floorHeight) { p.y = ex::add(floorHeight, r); q[i] = p; }
}

// velocity + floor friction (Solver.cpp:140-158)
__global__ void __launch_bounds__(kThreads) k_pbd_velocity(uint32_t n, const float4* __restrict__ q,
                                                           const float4* __restrict__ prev, float4* __restrict__ vel,
                                                           float dt, float damping, float friction, float floorHeight) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q[i], o = prev[i];
  float k = ex::sub(1.0f, damping);
  float vx = ex::div(ex::mul(k, ex::sub(p.x, o.x)), dt);
  float vy = ex::div(ex::mul(k, ex::sub(p.y, o.y)), dt);
  float vz = ex::div(ex::mul(k, ex::sub(p.z, o.z)), dt);
  if (ex::sub(p.y, o.w) <= floorHeight) {
    float planar = __fsqrt_rn(ex::add(ex::mul(vx, vx), ex::mul(vz, vz)));
    if (planar < 5.0f) { vx = 0.0f; vz = 0.0f; }
    else { float f = ex::sub(1.0f, friction); vx = ex::mul(vx, f); vz = ex::mul(vz, f); }
  }
  vel[i] = make_float4(vx, vy, vz, 0.0f);
}

// ------------------------------------------------------------------------------------------
// ordered constraint sweeps
struct PosOp {   // Constraint<1>::projectNodePositions with PositionConstraintProjection (Constraints.cpp:58-63)
  const uint32_t* ids; const uint32_t* tk; const float4* targetW;
  static constexpr int kNodes = 1;
  __device__ __forceinline__ void load(uint32_t e, uint32_t (&id)[4], uint32_t (&t)[4]) const { id[0] = ids[e]; t[0] = tk[e]; }
  __device__ __forceinline__ void run(uint32_t e, const uint32_t (&id)[4], float4* q) const {
    float4 p = __ldcg(q + id[0]);
    float4 tw = targetW[e];
    p.x = ex::add(p.x, ex::mul(tw.w, ex::sub(tw.x, p.x)));
    p.y = ex::add(p.y, ex::mul(tw.w, ex::sub(tw.y, p.y)));
    p.z = ex::add(p.z, ex::mul(tw.w, ex::sub(tw.z, p.z)));
    __stcg(q + id[0], p);
  }
};

struct DistOp {  // DistanceConstraintProjection (Constraints.cpp:11-37) + projectNodePositions
  const uint2* ids; const uint2* tk; const float2* restW;
  static constexpr int kNodes = 2;
  __device__ __forceinline__ void load(uint32_t e, uint32_t (&id)[4], uint32_t (&t)[4]) const {
    uint2 a = ids[e], b = tk[e]; id[0] = a.x; id[1] = a.y; t[0] = b.x; t[1] = b.y;
  }
  __device__ __forceinline__ void run(uint32_t e, const uint32_t (&id)[4], float4* q) const {
    float4 a4 = __ldcg(q + id[0]), b4 = __ldcg(q + id[1]);
    float2 rw = restW[e];
    V3 a = v3(a4), b = v3(b4);
    V3 diff = ex::sub(b, a);
    float dist = __fsqrt_rn(ex::dot3(diff, diff));
    V3 dir = v3(1.0f, 0.0f, 0.0f);
    if (dist > 0.00001f) dir = v3(ex::div(diff.x, dist), ex::div(diff.y, dist), ex::div(diff.z, dist));
    float disp = ex::sub(rw.x, dist);
    V3 p0 = ex::add(a, ex::scale(dir, -disp));       // projected[0] += -disp * dir
    // node 0: position += w (p0 - position); node 1: projected == position, += w * 0 leaves it unchanged
    a4.x = ex::add(a.x, ex::mul(rw.y, ex::sub(p0.x, a.x)));
    a4.y = ex::add(a.y, ex::mul(rw.y, ex::sub(p0.y, a.y)));
    a4.z = ex::add(a.z, ex::mul(rw.y, ex::sub(p0.z, a.z)));
    __stcg(q + id[0], a4);
  }
};

struct BendOp {  // BendConstraintProjection (Constraints.cpp:312-366) + projectNodePositions
  const uint4* ids; const uint4* tk; const float2* angleW;
  static constexpr int kNodes = 4;
  __device__ __forceinline__ void load(uint32_t e, uint32_t (&id)[4], uint32_t (&t)[4]) const {
    uint4 a = ids[e], b = tk[e];
    id[0] = a.x; id[1] = a.y; id[2] = a.z; id[3] = a.w; t[0] = b.x; t[1] = b.y; t[2] = b.z; t[3] = b.w;
  }
  __device__ __forceinline__ void run(uint32_t e, const uint32_t (&id)[4], float4* q) const {
    float4 n1_ = __ldcg(q + id[0]), n2_ = __ldcg(q + id[1]), n3_ = __ldcg(q + id[2]), n4_ = __ldcg(q + id[3]);
    float2 aw = angleW[e];
    V3 x1 = v3(n1_), x2 = v3(n2_), x3 = v3(n3_), x4 = v3(n4_);
    V3 p2 = ex::sub(x2, x1), p3 = ex::sub(x3, x1), p4 = ex::sub(x4, x1);
    V3 c23 = ex::cross3(p2, p3), c24 = ex::cross3(p2, p4);
    float l23 = __fsqrt_rn(ex::dot3(c23, c23)), l24 = __fsqrt_rn(ex::dot3(c24, c24));
    V3 n1 = v3(ex::div(c23.x, l23), ex::div(c23.y, l23), ex::div(c23.z, l23));
    V3 n2 = v3(ex::div(c24.x, l24), ex::div(c24.y, l24), ex::div(c24.z, l24));
    float d = ex::dot3(n1, n2);
    float d2 = ex::mul(d, d);
    // the reference's unqualified acos()/sqrt() are the double overloads: C and the numerator are rounded to float once
    float C = (float)(acos((double)d) - (double)aw.x);
    auto divv = [](V3 a, float s) { return v3(ex::div(a.x, s), ex::div(a.y, s), ex::div(a.z, s)); };
    V3 q3 = divv(ex::add(ex::cross3(p2, n2), ex::scale(ex::cross3(n1, p2), d)), l23);
    V3 q4 = divv(ex::add(ex::cross3(p2, n1), ex::scale(ex::cross3(n2, p2), d)), l24);
    V3 t3 = divv(ex::add(ex::cross3(p3, n2), ex::scale(ex::cross3(n1, p3), d)), l23);
    V3 t4 = divv(ex::add(ex::cross3(p4, n1), ex::scale(ex::cross3(n2, p4), d)), l24);
    V3 q2 = ex::sub(v3(-t3.x, -t3.y, -t3.z), t4);
    V3 q1 = ex::sub(ex::sub(v3(-q2.x, -q2.y, -q2.z), q3), q4);
    float wSum = ex::add(ex::add(ex::add(n1_.w, n2_.w), n3_.w), n4_.w);
    float qq = ex::add(ex::add(ex::add(ex::dot3(q1, q1), ex::dot3(q2, q2)), ex::dot3(q3, q3)), ex::dot3(q4, q4));
    float om = ex::sub(1.0f, d2);
    float num = (float)(sqrt((double)(om < 0.0f ? 0.0f : om)) * (double)C);  // glm::max(x, 0) keeps a NaN x
    if (qq < 0.00001f) return;  // projected == positions: position += w * 0
    const V3 qs[4] = {q1, q2, q3, q4};
    float4 nodes[4] = {n1_, n2_, n3_, n4_};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float s = ex::div(ex::mul(4.0f, nodes[k].w), wSum);
      // projected += -q * s * num / qq   (left to right)
      V3 dlt = v3(ex::div(ex::mul(ex::mul(-qs[k].x, s), num), qq), ex::div(ex::mul(ex::mul(-qs[k].y, s), num), qq),
                  ex::div(ex::mul(ex::mul(-qs[k].z, s), num), qq));
      V3 pos = v3(nodes[k]);
      V3 proj = ex::add(pos, dlt);
      nodes[k].x = ex::add(pos.x, ex::mul(aw.y, ex::sub(proj.x, pos.x)));
      nodes[k].y = ex::add(pos.y, ex::mul(aw.y, ex::sub(proj.y, pos.y)));
      nodes[k].z = ex::add(pos.z, ex::mul(aw.y, ex::sub(proj.z, pos.z)));
      __stcg(q + id[k], nodes[k]);
    }
  }
};

// Dataflow executor (same scheme as k_gs_dataflow in contact.cu): warps take chunks of 32 consecutive
// ops from a global counter, so every chunk below the newest is owned by a running warp and the earliest
// unfinished op is always runnable.
template <typename Op>
__global__ void __launch_bounds__(kSweepThreads) k_pbd_sweep(uint32_t nOps, Op op, float4* __restrict__ q,
                                                             uint32_t* __restrict__ nodeDone,
                                                             uint32_t* __restrict__ chunkCounter) {
  const int lane = threadIdx.x & 31;
  const uint32_t nChunks = (nOps + 31u) >> 5;
  while (true) {
    uint32_t chunk = 0;
    if (lane == 0) chunk = atomicAdd(chunkCounter, 1u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    if (chunk >= nChunks) break;
    uint32_t e = (chunk << 5) + (uint32_t)lane;
    bool pending = e < nOps;
    uint32_t id[4] = {0, 0, 0, 0}, tk[4] = {0, 0, 0, 0};
    if (pending) op.load(e, id, tk);
    while (__any_sync(0xffffffffu, pending)) {
      if (pending) {
        bool ready = true;
#pragma unroll
        for (int k = 0; k < Op::kNodes; ++k) ready = ready && ldAcquire(nodeDone + id[k]) == tk[k];
        if (ready) {
          op.run(e, id, q);
          __threadfence();
#pragma unroll
          for (int k = 0; k < Op::kNodes; ++k) stRelease(nodeDone + id[k], tk[k] + 1u);
          pending = false;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// node hash
__global__ void k_pbd_init(int* bbox, uint32_t* flags) {
  bbox[0] = bbox[1] = bbox[2] = 0x7fffffff;
  bbox[3] = bbox[4] = bbox[5] = (int)0x80000000;
  bbox[6] = 0; bbox[7] = 0;
  flags[0] = 0; flags[1] = 0;
}

__global__ void __launch_bounds__(kThreads) k_node_ranges(uint32_t n, const float4* __restrict__ q,
                                                          const float4* __restrict__ prev, float scale,
                                                          int4* __restrict__ nodeMin, uint32_t* __restrict__ nodeLen,
                                                          uint32_t* __restrict__ cnt, float4* __restrict__ q0,
                                                          int* __restrict__ bbox) {
  __shared__ int sb[8];
  if (threadIdx.x < 3) sb[threadIdx.x] = 0x7fffffff;
  else if (threadIdx.x < 6) sb[threadIdx.x] = (int)0x80000000;
  else if (threadIdx.x < 8) sb[threadIdx.x] = 0;
  __syncthreads();
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float4 p = q[i];
    q0[i] = p;
    int mx, my, mz; unsigned lx, ly, lz; bool bad;
    ex::nodeCellRange(v3(p), prev[i].w, scale, mx, my, mz, lx, ly, lz, bad);
    if (bad) sb[6] = 1;
    nodeMin[i] = make_int4(mx, my, mz, 0);
    nodeLen[i] = lx | (ly << 8) | (lz << 16);
    uint32_t cells = lx * ly * lz;
    cnt[i] = cells;
    if (cells) {
      atomicMin(&sb[0], mx); atomicMin(&sb[1], my); atomicMin(&sb[2], mz);
      atomicMax(&sb[3], mx + (int)lx - 1); atomicMax(&sb[4], my + (int)ly - 1); atomicMax(&sb[5], mz + (int)lz - 1);
    }
  }
  __syncthreads();
  if (threadIdx.x < 3) { if (sb[threadIdx.x] != 0x7fffffff) atomicMin(bbox + threadIdx.x, sb[threadIdx.x]); }
  else if (threadIdx.x < 6) { if (sb[threadIdx.x] != (int)0x80000000) atomicMax(bbox + threadIdx.x, sb[threadIdx.x]); }
  else if (threadIdx.x < 8) { if (sb[threadIdx.x]) atomicExch(bbox + threadIdx.x, 1); }
}

struct NodeKeyPack { int minX, minY, minZ, maxX, maxY, maxZ; int bitsY, bitsZ; };

__device__ __forceinline__ uint64_t packCell(const NodeKeyPack& kp, int x, int y, int z) {
  return ((uint64_t)(uint32_t)(x - kp.minX) << (kp.bitsY + kp.bitsZ)) | ((uint64_t)(uint32_t)(y - kp.minY) << kp.bitsZ) |
         (uint64_t)(uint32_t)(z - kp.minZ);
}

__global__ void __launch_bounds__(kThreads) k_node_pairs(uint32_t n, const int4* __restrict__ nodeMin,
                                                         const uint32_t* __restrict__ nodeLen,
                                                         const uint32_t* __restrict__ off, NodeKeyPack kp,
                                                         uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t len = nodeLen[i];
  uint32_t lx = len & 255u, ly = (len >> 8) & 255u, lz = (len >> 16) & 255u;
  if (!(lx * ly * lz)) return;
  int4 m = nodeMin[i];
  uint32_t k = off[i];
  for (uint32_t dx = 0; dx < lx; ++dx)
    for (uint32_t dy = 0; dy < ly; ++dy)
      for (uint32_t dz = 0; dz < lz; ++dz, ++k) {
        keys[k] = packCell(kp, m.x + (int)dx, m.y + (int)dy, m.z + (int)dz);
        vals[k] = i;
      }
}

__global__ void __launch_bounds__(kThreads) k_pbd_heads(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                        uint32_t* __restrict__ heads) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > nPairs) return;
  heads[j] = (j < nPairs && (j == 0 || keys[j] != keys[j - 1])) ? 1u : 0u;
}

// cellStart[c], cellKey[c] for every distinct key (heads holds the exclusive scan of the head flags)
__global__ void __launch_bounds__(kThreads) k_pbd_cells(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                        const uint32_t* __restrict__ headScan,
                                                        uint32_t* __restrict__ cellStart, uint64_t* __restrict__ cellKey) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nPairs) return;
  bool head = (j == 0 || keys[j] != keys[j - 1]);
  uint32_t idx = headScan[j] + (head ? 1u : 0u) - 1u;
  if (head) { cellStart[idx] = (uint32_t)j; cellKey[idx] = keys[j]; }
  if (j == nPairs - 1) cellStart[idx + 1] = (uint32_t)nPairs;
}

__device__ __forceinline__ int findCell(const uint64_t* __restrict__ cellKey, uint32_t nCells, uint64_t key) {
  uint32_t lo = 0, hi = nCells;
  while (lo < hi) {
    uint32_t mid = (lo + hi) >> 1;
    uint64_t k = cellKey[mid];
    if (k < key) lo = mid + 1; else hi = mid;
  }
  return (lo < nCells && cellKey[lo] == key) ? (int)lo : -1;
}

// ------------------------------------------------------------------------------------------
// visit list: one thread per node, cells x-major / y / z (the reference's dx,dy,dz order), members ascending
template <bool WRITE>
__global__ void __launch_bounds__(kThreads) k_pbd_visits(uint32_t n, const float4* __restrict__ q0,
                                                         const float4* __restrict__ prev, float scale, float delta,
                                                         NodeKeyPack kp, const uint64_t* __restrict__ cellKey,
                                                         uint32_t nCells, const uint32_t* __restrict__ cellStart,
                                                         const uint32_t* __restrict__ member,
                                                         uint32_t* __restrict__ visCnt /* scanned when WRITE */,
                                                         uint4* __restrict__ visits) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float4 p = q0[i];
  float ri = prev[i].w;
  float R = ri + 0.5f + delta;
  int lo[3], hi[3];
  const float pc[3] = {p.x, p.y, p.z};
  const int bmin[3] = {kp.minX, kp.minY, kp.minZ}, bmax[3] = {kp.maxX, kp.maxY, kp.maxZ};
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    float l = floorf((pc[a] - R) / scale) - 1.0f, h = ceilf((pc[a] + R) / scale) + 1.0f;
    l = fmaxf(l, (float)bmin[a]); h = fminf(h, (float)bmax[a]);
    lo[a] = (int)l; hi[a] = (int)h;
  }
  uint32_t total = 0, out = WRITE ? visCnt[i] : 0u;
  for (int x = lo[0]; x <= hi[0]; ++x)
    for (int y = lo[1]; y <= hi[1]; ++y)
      for (int z = lo[2]; z <= hi[2]; ++z) {
        uint64_t key = packCell(kp, x, y, z);
        int c = findCell(cellKey, nCells, key);
        if (c < 0) continue;
        uint32_t s = cellStart[c], e = cellStart[c + 1];
        for (uint32_t m = s; m < e; ++m) {
          uint32_t j = member[m];
          float4 pj = q0[j];
          float rj = prev[j].w;
          float dx = pj.x - p.x, dy = pj.y - p.y, dz = pj.z - p.z;
          float reach = ri + rj + 2.0f * delta;
          if (dx * dx + dy * dy + dz * dz >= reach * reach * 1.0001f) continue;
          if (WRITE) {
            uint32_t first = total == 0 ? 0x80000000u : 0u;
            visits[out + total] = make_uint4(i, j, (uint32_t)key, (uint32_t)(key >> 32) | first);
          }
          ++total;
        }
      }
  if (!WRITE) visCnt[i] = total;
}

// (node, 2 * visit + slot) incidence pairs in visit order; self visits use one slot
__global__ void __launch_bounds__(kThreads) k_pbd_inc_emit(uint32_t nVis, uint32_t n, const uint4* __restrict__ visits,
                                                           uint64_t* __restrict__ keys, uint32_t* __restrict__ vals,
                                                           uint32_t* __restrict__ incCount) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nVis) return;
  uint4 v = visits[e];
  keys[2ull * e] = v.x; vals[2ull * e] = 2u * e;
  atomicAdd(incCount + v.x, 1u);
  if (v.y != v.x) { keys[2ull * e + 1] = v.y; atomicAdd(incCount + v.y, 1u); }
  else { keys[2ull * e + 1] = n; atomicAdd(incCount + n, 1u); }  // dummy node n collects the unused slots
  vals[2ull * e + 1] = 2u * e + 1u;
}

__global__ void __launch_bounds__(kThreads) k_pbd_tickets(uint64_t nInc, const uint64_t* __restrict__ sortedNode,
                                                          const uint32_t* __restrict__ inc,
                                                          const uint32_t* __restrict__ incPtr, uint32_t* __restrict__ ticket) {
  uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nInc) return;
  ticket[inc[k]] = (uint32_t)k - incPtr[(uint32_t)sortedNode[k]];
}

// node-node response sweep (Solver.cpp:85-111)
__global__ void __launch_bounds__(kSweepThreads) k_pbd_collide(uint32_t nVis, const uint4* __restrict__ visits,
                                                               const uint2* __restrict__ ticket, float4* __restrict__ q,
                                                               const float4* __restrict__ prev, float4* __restrict__ turnStart,
                                                               float scale, NodeKeyPack kp, const float4* __restrict__ q0,
                                                               float delta, uint32_t* __restrict__ flags,
                                                               uint32_t* __restrict__ nodeDone,
                                                               uint32_t* __restrict__ chunkCounter) {
  const int lane = threadIdx.x & 31;
  const uint32_t nChunks = (nVis + 31u) >> 5;
  const uint64_t maskZ = (1ull << kp.bitsZ) - 1ull, maskY = (1ull << kp.bitsY) - 1ull;
  while (true) {
    uint32_t chunk = 0;
    if (lane == 0) chunk = atomicAdd(chunkCounter, 1u);
    chunk = __shfl_sync(0xffffffffu, chunk, 0);
    if (chunk >= nChunks) break;
    uint32_t e = (chunk << 5) + (uint32_t)lane;
    bool pending = e < nVis;
    uint4 v = make_uint4(0, 0, 0, 0);
    uint2 tk = make_uint2(0, 0);
    if (pending) { v = visits[e]; tk = ticket[e]; }
    const uint32_t i = v.x, j = v.y;
    const bool self = i == j, first = (v.w & 0x80000000u) != 0u;
    while (__any_sync(0xffffffffu, pending)) {
      if (pending) {
        bool ready = ldAcquire(nodeDone + i) == tk.x && (self || ldAcquire(nodeDone + j) == tk.y);
        if (ready) {
          float4 pi = __ldcg(q + i);
          float4 ts;
          if (first) { ts = pi; __stcg(turnStart + i, pi); } else ts = __ldcg(turnStart + i);
          float ri = prev[i].w;
          int mx, my, mz; unsigned lx, ly, lz; bool bad;
          ex::nodeCellRange(v3(ts), ri, scale, mx, my, mz, lx, ly, lz, bad);
          uint64_t key = ((uint64_t)(v.w & 0x7fffffffu) << 32) | (uint64_t)v.z;
          int cz = (int)(key & maskZ) + kp.minZ, cy = (int)((key >> kp.bitsZ) & maskY) + kp.minY,
              cx = (int)(key >> (kp.bitsY + kp.bitsZ)) + kp.minX;
          bool inRange = cx >= mx && cx < mx + (int)lx && cy >= my && cy < my + (int)ly && cz >= mz && cz < mz + (int)lz;
          if (inRange) {
            float4 pj = self ? pi : __ldcg(q + j);
            float rj = self ? ri : prev[j].w;
            V3 diff = ex::sub(v3(pj), v3(pi));
            float dist = __fsqrt_rn(ex::dot3(diff, diff));
            float disp = ex::sub(ex::add(ri, rj), dist);
            if (disp > 0.0f) {
              V3 dir = v3(1.0f, 0.0f, 0.0f);
              if (dist > 0.00001f) dir = v3(ex::div(diff.x, dist), ex::div(diff.y, dist), ex::div(diff.z, dist));
              float wSum = ex::add(pi.w, pj.w);
              float ka = ex::mul(0.85f, -disp), kb = ex::mul(0.85f, disp);
              V3 da = v3(ex::div(ex::mul(ex::mul(ka, dir.x), pi.w), wSum), ex::div(ex::mul(ex::mul(ka, dir.y), pi.w), wSum),
                         ex::div(ex::mul(ex::mul(ka, dir.z), pi.w), wSum));
              V3 db = v3(ex::div(ex::mul(ex::mul(kb, dir.x), pj.w), wSum), ex::div(ex::mul(ex::mul(kb, dir.y), pj.w), wSum),
                         ex::div(ex::mul(ex::mul(kb, dir.z), pj.w), wSum));
              pi.x = ex::add(pi.x, da.x); pi.y = ex::add(pi.y, da.y); pi.z = ex::add(pi.z, da.z);
              // the visit list was pruned assuming no node strays further than delta from its position at hash
              // build, at ANY time during the sweep: check every write (the host redoes the pass if violated)
              if (self) {  // both updates land on the same node, one after the other (net zero up to rounding)
                pi.x = ex::add(pi.x, db.x); pi.y = ex::add(pi.y, db.y); pi.z = ex::add(pi.z, db.z);
                __stcg(q + i, pi);
              } else {
                pj.x = ex::add(pj.x, db.x); pj.y = ex::add(pj.y, db.y); pj.z = ex::add(pj.z, db.z);
                __stcg(q + i, pi); __stcg(q + j, pj);
              }
              float4 bi = q0[i];
              float moved = fmaxf(fmaxf(fabsf(pi.x - bi.x), fabsf(pi.y - bi.y)), fabsf(pi.z - bi.z));
              if (!self) {
                float4 bj = q0[j];
                moved = fmaxf(moved, fmaxf(fmaxf(fabsf(pj.x - bj.x), fabsf(pj.y - bj.y)), fabsf(pj.z - bj.z)));
              }
              if (!(moved <= delta)) flags[0] = 1u;
            }
          }
          __threadfence();
          stRelease(nodeDone + i, tk.x + 1u);
          if (!self) stRelease(nodeDone + j, tk.y + 1u);
          pending = false;
        }
      }
    }
  }
}

// ------------------------------------------------------------------------------------------
// Colour-batched node-node response (the north_star's "graph-coloured Jacobi-free batches"), opt-in.
//
// The reference's response is ONE sequential sweep: node i's visits modify its partners before their own turn, so on
// a scene whose contact graph is a long chain (a coiled rope: every node touches its neighbours) the dependency chain
// of the ordered executor above is as long as the visit list — exact, and serial (measured: seconds per tick beyond a
// few thousand nodes).  This mode gives up the reference's ORDER, not its operation: the distinct overlapping pairs of
// the visit list are edge-coloured (no two pairs of a colour share a node), colours run one after the other, and a
// pair receives the reference's response (push apart by 0.85 x overlap, mass weighted, Solver.cpp:100-110) as many
// times as the reference would have visited it (once per shared cell from either side), each time on the updated
// positions.  Deterministic (integer atomics only, fixed priorities); results differ from the reference's like a
// different visiting order does (SURVEY F4), so the parity tests run the ordered executor and this mode is held to
// physical properties (tests/test_pbd_gpu.py).
__device__ __forceinline__ uint32_t pairPriority(uint32_t p) {  // fixed pseudo-random priority: long chains colour in O(log n) rounds
  uint32_t h = p * 2654435761u;
  h ^= h >> 15; h *= 2246822519u; h ^= h >> 13;
  return h;
}

// distinct partners j > i of node i in its visit range, with the number of visits (shared cells)
template <bool WRITE>
__global__ void __launch_bounds__(kThreads) k_pbd_pairs(uint32_t n, const uint32_t* __restrict__ visOff, const uint4* __restrict__ visits,
                                                        uint32_t* __restrict__ pairCnt /* scanned when WRITE */, uint4* __restrict__ pairs) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint32_t s = visOff[i], e = visOff[i + 1];
  uint32_t total = 0, out = WRITE ? pairCnt[i] : 0u;
  for (uint32_t k = s; k < e; ++k) {
    const uint32_t j = visits[k].y;
    if (j <= i) continue;
    bool seen = false;
    for (uint32_t m = s; m < k && !seen; ++m) seen = visits[m].y == j;
    if (seen) continue;
    if (WRITE) {
      uint32_t cnt = 1;
      for (uint32_t m = k + 1; m < e; ++m) cnt += visits[m].y == j ? 1u : 0u;
      pairs[out + total] = make_uint4(i, j, 2u * cnt, 0u);   // the partner visits the pair as often from its side
    }
    ++total;
  }
  if (!WRITE) pairCnt[i] = total;
}

__global__ void __launch_bounds__(kThreads) k_pbd_color_propose(uint32_t nP, const uint4* __restrict__ pairs,
                                                                const uint32_t* __restrict__ color, uint32_t* __restrict__ nodeMinPrio) {
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nP || color[p] != 0xffffffffu) return;
  const uint32_t pr = pairPriority(p);
  atomicMin(nodeMinPrio + pairs[p].x, pr);
  atomicMin(nodeMinPrio + pairs[p].y, pr);
}

// a pair whose priority is the smallest among the uncoloured pairs at BOTH its nodes takes the lowest colour free at both
// (no other pair touches either node in this round, so the masks are updated without atomics)
__global__ void __launch_bounds__(kThreads) k_pbd_color_commit(uint32_t nP, const uint4* __restrict__ pairs, uint32_t* __restrict__ color,
                                                               const uint32_t* __restrict__ nodeMinPrio,
                                                               unsigned long long* __restrict__ nodeMask, uint32_t* __restrict__ stat) {
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nP || color[p] != 0xffffffffu) return;
  const uint32_t a = pairs[p].x, b = pairs[p].y, pr = pairPriority(p);
  if (nodeMinPrio[a] == pr && nodeMinPrio[b] == pr) {
    const unsigned long long used = nodeMask[a] | nodeMask[b];
    const int c = __ffsll((long long)~used) - 1;   // -1: all 64 colours taken at these nodes (a node overlapping > 32 others)
    if (c >= 0) {
      color[p] = (uint32_t)c;
      nodeMask[a] |= 1ull << c; nodeMask[b] |= 1ull << c;
      atomicMax(stat + 1, (uint32_t)c + 1u);
      return;
    }
    // all 64 colours taken at its nodes (a node overlapping dozens of others: a collapsed scene): the pair gets a colour
    // of its own after the regular ones; the host gives up beyond 256 of them
    const uint32_t extra = atomicAdd(stat + 2, 1u);
    color[p] = 64u + extra;
    return;
  }
  atomicAdd(stat, 1u);  // still uncoloured after this round
}

__global__ void __launch_bounds__(kThreads) k_pbd_apply_color(uint32_t nP, uint32_t c, const uint4* __restrict__ pairs,
                                                              const uint32_t* __restrict__ color, float4* __restrict__ q,
                                                              const float4* __restrict__ prev, const float4* __restrict__ q0, float delta,
                                                              uint32_t* __restrict__ flags) {
  uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nP || color[p] != c) return;
  const uint4 pr = pairs[p];
  float4 pi = q[pr.x], pj = q[pr.y];
  const float ri = prev[pr.x].w, rj = prev[pr.y].w;
  const float wSum = pi.w + pj.w;
  bool moved = false;
  for (uint32_t k = 0; k < pr.z; ++k) {  // Solver.cpp:95-110, once per visit the reference makes
    const float dx = pj.x - pi.x, dy = pj.y - pi.y, dz = pj.z - pi.z;
    const float dist = sqrtf(dx * dx + dy * dy + dz * dz);
    const float disp = ri + rj - dist;
    if (!(disp > 0.0f)) break;
    float nx = 1.0f, ny = 0.0f, nz = 0.0f;
    if (dist > 0.00001f) { nx = dx / dist; ny = dy / dist; nz = dz / dist; }
    const float ka = -0.85f * disp * pi.w / wSum, kb = 0.85f * disp * pj.w / wSum;
    pi.x += ka * nx; pi.y += ka * ny; pi.z += ka * nz;
    pj.x += kb * nx; pj.y += kb * ny; pj.z += kb * nz;
    moved = true;
  }
  if (!moved) return;
  q[pr.x] = pi; q[pr.y] = pj;
  const float4 bi = q0[pr.x], bj = q0[pr.y];
  const float far = fmaxf(fmaxf(fmaxf(fabsf(pi.x - bi.x), fabsf(pi.y - bi.y)), fabsf(pi.z - bi.z)),
                          fmaxf(fmaxf(fabsf(pj.x - bj.x), fabsf(pj.y - bj.y)), fabsf(pj.z - bj.z)));
  if (!(far <= delta)) flags[0] = 1u;   // the pair list was pruned assuming no node strays further than delta
}

// ------------------------------------------------------------------------------------------
#define PCHECK(expr)                                                              \
  do {                                                                            \
    cudaError_t _e = (expr);                                                      \
    if (_e != cudaSuccess) return failCuda(s, _e, #expr, __LINE__);               \
  } while (0)

static int bitsFor(int64_t span) {
  int b = 1;
  while ((int64_t(1) << b) <= span) ++b;
  return b;
}

template <typename T>
static void hostTickets(const std::vector<uint32_t>& ids, int nodesPerOp, uint32_t nNodes, std::vector<uint32_t>& tk) {
  std::vector<uint32_t> seen(nNodes, 0);
  tk.resize(ids.size());
  for (size_t e = 0; e < ids.size() / nodesPerOp; ++e)
    for (int k = 0; k < nodesPerOp; ++k) tk[e * nodesPerOp + k] = seen[ids[e * nodesPerOp + k]]++;
  (void)sizeof(T);
}

static int buildPbd(PiesB200Solver* s, PbdWork& w) {
  const HostScene& sc = s->scene;
  cudaStream_t st = s->stream;
  const uint32_t n = sc.nodeCount();
  w.nPos = (uint32_t)sc.posW.size(); w.nDist = (uint32_t)sc.distW.size(); w.nBend = (uint32_t)sc.bendW.size();
  std::vector<uint32_t> tk;
  // A bend op touching the same node twice would wait on itself; the factories never emit one.
  hostTickets<int>(sc.posId, 1, n, tk);
  PCHECK(w.posIds.upload(sc.posId.data(), sc.posId.size(), st)); PCHECK(w.posTk.upload(tk.data(), tk.size(), st));
  std::vector<float4> ptw(w.nPos);
  for (uint32_t i = 0; i < w.nPos; ++i) ptw[i] = make_float4(sc.posTarget[3 * i], sc.posTarget[3 * i + 1], sc.posTarget[3 * i + 2], sc.posW[i]);
  PCHECK(w.posTargetW.upload(ptw.data(), ptw.size(), st));
  PCHECK(cudaStreamSynchronize(st));
  hostTickets<int>(sc.distId, 2, n, tk);
  PCHECK(w.distIds.upload(reinterpret_cast<const uint2*>(sc.distId.data()), w.nDist, st));
  PCHECK(w.distTk.upload(reinterpret_cast<const uint2*>(tk.data()), w.nDist, st));
  std::vector<float2> drw(w.nDist);
  for (uint32_t i = 0; i < w.nDist; ++i) drw[i] = make_float2(sc.distRest[i], sc.distW[i]);
  PCHECK(w.distRestW.upload(drw.data(), drw.size(), st));
  PCHECK(cudaStreamSynchronize(st));
  for (uint32_t e = 0; e < w.nDist; ++e)
    if (sc.distId[2 * e] == sc.distId[2 * e + 1]) return fail(s, PIES_B200_EINVAL, "distance constraint with identical end nodes");
  for (uint32_t e = 0; e < w.nBend; ++e)
    for (int a = 0; a < 4; ++a)
      for (int b = a + 1; b < 4; ++b)
        if (sc.bendId[4 * e + a] == sc.bendId[4 * e + b]) return fail(s, PIES_B200_EINVAL, "bend constraint with a repeated node");
  hostTickets<int>(sc.bendId, 4, n, tk);
  PCHECK(w.bendIds.upload(reinterpret_cast<const uint4*>(sc.bendId.data()), w.nBend, st));
  PCHECK(w.bendTk.upload(reinterpret_cast<const uint4*>(tk.data()), w.nBend, st));
  std::vector<float2> baw(w.nBend);
  for (uint32_t i = 0; i < w.nBend; ++i) baw[i] = make_float2(sc.bendAngle[i], sc.bendW[i]);
  PCHECK(w.bendAngleW.upload(baw.data(), baw.size(), st));
  PCHECK(cudaStreamSynchronize(st));
  PCHECK(w.nodeDone.reserve(n + 2)); PCHECK(w.counters.reserve(64));
  PCHECK(w.nodeMin.reserve(n)); PCHECK(w.nodeLen.reserve(n)); PCHECK(w.cnt.reserve(n + 2)); PCHECK(w.visCnt.reserve(n + 2));
  PCHECK(w.q0.reserve(n)); PCHECK(w.turnStart.reserve(n)); PCHECK(w.bbox.reserve(8)); PCHECK(w.flags.reserve(4));
  PCHECK(w.incPtr.reserve(n + 3));
  if (!w.host) PCHECK(cudaMallocHost(&w.host, 16 * sizeof(int)));
  w.builtVersion = sc.topologyVersion;
  return PIES_B200_OK;
}

template <typename Op>
static int sweep(PiesB200Solver* s, PbdWork& w, uint32_t nOps, Op op) {
  if (!nOps) return PIES_B200_OK;
  cudaStream_t st = s->stream;
  if (w.countersUsed == 64) { PCHECK(cudaMemsetAsync(w.counters.p, 0, 64 * sizeof(uint32_t), st)); w.countersUsed = 0; }
  PCHECK(cudaMemsetAsync(w.nodeDone.p, 0, (size_t)(s->n + 2) * sizeof(uint32_t), st));
  uint32_t chunks = (nOps + 31u) / 32u;
  int grid = (int)std::min<uint32_t>(kNumSMs * 4, (chunks + kSweepThreads / 32 - 1) / (kSweepThreads / 32));
  k_pbd_sweep<Op><<<grid, kSweepThreads, 0, st>>>(nOps, op, s->q.p, w.nodeDone.p, w.counters.p + w.countersUsed);
  ++w.countersUsed; ++s->launches;
  return PIES_B200_OK;
}

// Hash rebuild (Solver.cpp:81-82): fills the sorted (cell, node) table; kp / w.nCells / w.nPairs describe it.
static int buildNodeHash(PiesB200Solver* s, PbdWork& w, NodeKeyPack& kp) {
  cudaStream_t st = s->stream;
  const uint32_t n = s->n;
  const float scale = s->opt.gridSpacing;
  k_pbd_init<<<1, 1, 0, st>>>(w.bbox.p, w.flags.p); ++s->launches;
  PCHECK(cudaMemsetAsync(w.cnt.p + n, 0, 2 * sizeof(uint32_t), st));
  k_node_ranges<<<gridFor(n, kThreads), kThreads, 0, st>>>(n, s->q.p, s->prev.p, scale, w.nodeMin.p, w.nodeLen.p, w.cnt.p,
                                                          w.q0.p, w.bbox.p); ++s->launches;
  PCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(n + 3, 1024))));
  s->launches += launchExclusiveScan(st, w.cnt.p, n + 1, w.scanScratch.p);
  PCHECK(cudaMemcpyAsync(w.host, w.bbox.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, st));
  PCHECK(cudaMemcpyAsync(w.host + 8, w.cnt.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  PCHECK(cudaStreamSynchronize(st));
  if (w.host[6]) { s->simFailed = true; return fail(s, PIES_B200_ERANGE, "non-finite or out-of-range positions reached the node hash"); }
  const uint64_t nPairs = (uint32_t)w.host[8];
  w.nPairs = nPairs; w.nCells = 0;
  if (!nPairs) return PIES_B200_OK;
  kp = NodeKeyPack{w.host[0], w.host[1], w.host[2], w.host[3], w.host[4], w.host[5], 0, 0};
  int bx = bitsFor((int64_t)kp.maxX - kp.minX), by = bitsFor((int64_t)kp.maxY - kp.minY), bz = bitsFor((int64_t)kp.maxZ - kp.minZ);
  kp.bitsY = by; kp.bitsZ = bz;
  if (bx + by + bz > 62) { s->simFailed = true; return fail(s, PIES_B200_ERANGE, "node hash extent exceeds 62 key bits"); }
  w.keyPack[0] = kp.minX; w.keyPack[1] = kp.minY; w.keyPack[2] = kp.minZ; w.keyPack[3] = by; w.keyPack[4] = bz;
  PCHECK(w.keys.reserve(nPairs)); PCHECK(w.tmpKeys.reserve(nPairs)); PCHECK(w.vals.reserve(nPairs)); PCHECK(w.tmpVals.reserve(nPairs));
  PCHECK(w.heads.reserve(nPairs + 2)); PCHECK(w.cellStart.reserve(nPairs + 2)); PCHECK(w.cellKey.reserve(nPairs + 2));
  PCHECK(w.sortHist.reserve(sortHistBytes(nPairs) / 4 + 4));
  PCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(nPairs + 2, n + 3))));
  k_node_pairs<<<gridFor(n, kThreads), kThreads, 0, st>>>(n, w.nodeMin.p, w.nodeLen.p, w.cnt.p, kp, w.keys.p, w.vals.p); ++s->launches;
  s->launches += launchSortPairs(st, nPairs, w.keys.p, w.vals.p, w.tmpKeys.p, w.tmpVals.p, w.sortHist.p, bx + by + bz);
  k_pbd_heads<<<gridFor(nPairs + 1, kThreads), kThreads, 0, st>>>(nPairs, w.keys.p, w.heads.p); ++s->launches;
  s->launches += launchExclusiveScan(st, w.heads.p, nPairs + 1, w.scanScratch.p);
  k_pbd_cells<<<gridFor(nPairs, kThreads), kThreads, 0, st>>>(nPairs, w.keys.p, w.heads.p, w.cellStart.p, w.cellKey.p); ++s->launches;
  PCHECK(cudaMemcpyAsync(w.host + 9, w.heads.p + nPairs, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  PCHECK(cudaStreamSynchronize(st));
  w.nCells = (uint32_t)w.host[9];
  return PIES_B200_OK;
}

// One iteration's hash rebuild + ordered node-node response (Solver.cpp:81-130).
static int collideNodes(PiesB200Solver* s, PbdWork& w) {
  cudaStream_t st = s->stream;
  const uint32_t n = s->n;
  const float scale = s->opt.gridSpacing;
  NodeKeyPack kp{};
  int rc = buildNodeHash(s, w, kp);
  if (rc) return rc;
  const uint64_t nPairs = w.nPairs;
  const uint32_t nCells = w.nCells;
  if (!nPairs) return PIES_B200_OK;

  if (w.delta <= 0.0f) w.delta = 0.125f * scale;
  for (int attempt = 0; attempt < 8; ++attempt) {
    const float delta = w.delta;
    PCHECK(cudaMemsetAsync(w.visCnt.p + n, 0, 2 * sizeof(uint32_t), st));
    k_pbd_visits<false><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, w.q0.p, s->prev.p, scale, delta, kp, w.cellKey.p, nCells,
                                                                  w.cellStart.p, w.vals.p, w.visCnt.p, nullptr); ++s->launches;
    s->launches += launchExclusiveScan(st, w.visCnt.p, n + 1, w.scanScratch.p);
    PCHECK(cudaMemcpyAsync(w.host + 10, w.visCnt.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCHECK(cudaStreamSynchronize(st));
    const uint32_t nVis = (uint32_t)w.host[10];
    if (!nVis) return PIES_B200_OK;
    const uint64_t nInc = 2ull * nVis;
    PCHECK(w.visits.reserve(nVis)); PCHECK(w.visTk.reserve(nVis));
    PCHECK(w.incKeys.reserve(nInc)); PCHECK(w.incTmpKeys.reserve(nInc)); PCHECK(w.incVals.reserve(nInc)); PCHECK(w.incTmpVals.reserve(nInc));
    PCHECK(w.sortHist.reserve(sortHistBytes(std::max<uint64_t>(nInc, nPairs)) / 4 + 4));
    PCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(std::max<uint64_t>(nInc, nPairs) + 2, n + 3))));
    k_pbd_visits<true><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, w.q0.p, s->prev.p, scale, delta, kp, w.cellKey.p, nCells,
                                                                 w.cellStart.p, w.vals.p, w.visCnt.p, w.visits.p); ++s->launches;
    if (s->tune.reserved & 1024u) {
      // ---- colour-batched response (see k_pbd_pairs ...): distinct pairs, edge colouring, one launch per colour
      PCHECK(w.pairCnt.reserve(n + 2)); PCHECK(w.nodeMinPrio.reserve(n + 1)); PCHECK(w.nodeMask.reserve(n + 1)); PCHECK(w.colorStat.reserve(4));
      PCHECK(cudaMemsetAsync(w.pairCnt.p + n, 0, 2 * sizeof(uint32_t), st));
      k_pbd_pairs<false><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, w.visCnt.p, w.visits.p, w.pairCnt.p, nullptr); ++s->launches;
      s->launches += launchExclusiveScan(st, w.pairCnt.p, n + 1, w.scanScratch.p);
      PCHECK(cudaMemcpyAsync(w.host + 12, w.pairCnt.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      PCHECK(cudaStreamSynchronize(st));
      const uint32_t nP = (uint32_t)w.host[12];
      bool fallBack = false;
      if (nP) {
        PCHECK(w.pairs.reserve(nP)); PCHECK(w.pairColor.reserve(nP));
        k_pbd_pairs<true><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, w.visCnt.p, w.visits.p, w.pairCnt.p, w.pairs.p); ++s->launches;
        PCHECK(cudaMemsetAsync(w.pairColor.p, 0xff, (size_t)nP * sizeof(uint32_t), st));
        PCHECK(cudaMemsetAsync(w.nodeMask.p, 0, (size_t)(n + 1) * sizeof(unsigned long long), st));
        PCHECK(cudaMemsetAsync(w.colorStat.p, 0, 4 * sizeof(uint32_t), st));
        uint32_t left = nP, colors = 0, leftOut = 0;
        for (int batch = 0; batch < 64 && left; ++batch) {   // 16 rounds per host read; a handful of batches at most
          for (int round = 0; round < 16; ++round) {
            PCHECK(cudaMemsetAsync(w.nodeMinPrio.p, 0xff, (size_t)(n + 1) * sizeof(uint32_t), st));
            PCHECK(cudaMemsetAsync(w.colorStat.p, 0, sizeof(uint32_t), st));
            k_pbd_color_propose<<<gridFor(nP, kThreads), kThreads, 0, st>>>(nP, w.pairs.p, w.pairColor.p, w.nodeMinPrio.p);
            k_pbd_color_commit<<<gridFor(nP, kThreads), kThreads, 0, st>>>(nP, w.pairs.p, w.pairColor.p, w.nodeMinPrio.p, w.nodeMask.p,
                                                                          w.colorStat.p);
            s->launches += 2;
          }
          PCHECK(cudaMemcpyAsync(w.host + 12, w.colorStat.p, 3 * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
          PCHECK(cudaStreamSynchronize(st));
          left = (uint32_t)w.host[12]; colors = (uint32_t)w.host[13]; leftOut = (uint32_t)w.host[14];
        }
        if (left != 0 || leftOut > 256) {
          // never silently fall back to the ordered executor here: on the scenes this mode exists for it would not return
          s->simFailed = true;
          return fail(s, PIES_B200_ERANGE, "PBD colour batches: the contact graph could not be coloured (a node overlaps more than 64 others: the scene has collapsed)");
        }
        if (leftOut) colors = 64u + leftOut;
        if (!fallBack) {
          for (uint32_t c = 0; c < colors; ++c) {
            if (c >= (uint32_t)w.host[13] && c < 64u) continue;   // unused regular colours below the private ones
            k_pbd_apply_color<<<gridFor(nP, kThreads), kThreads, 0, st>>>(nP, c, w.pairs.p, w.pairColor.p, s->q.p, s->prev.p, w.q0.p,
                                                                         delta, w.flags.p);
            ++s->launches;
          }
          PCHECK(cudaMemcpyAsync(w.host + 11, w.flags.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
          PCHECK(cudaStreamSynchronize(st));
          w.visitsLastTick += nVis;
          if (getenv("PIES_DEBUG_PBD"))
            std::fprintf(stderr, "[pbd] colour-batched: visits %u pairs %u colours %u delta %g attempt %d -> %s\n", nVis, nP, colors, delta,
                         attempt, w.host[11] ? "redo" : "ok");
          if (!w.host[11]) return PIES_B200_OK;
          PCHECK(cudaMemcpyAsync(s->q.p, w.q0.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, st));
          PCHECK(cudaMemsetAsync(w.flags.p, 0, sizeof(uint32_t), st));
          w.delta *= 2.0f;
          continue;
        }
      } else {
        w.visitsLastTick += nVis;
        return PIES_B200_OK;   // only self visits: net zero
      }
    }
    PCHECK(cudaMemsetAsync(w.incPtr.p, 0, (size_t)(n + 3) * sizeof(uint32_t), st));
    k_pbd_inc_emit<<<gridFor(nVis, kThreads), kThreads, 0, st>>>(nVis, n, w.visits.p, w.incKeys.p, w.incVals.p, w.incPtr.p); ++s->launches;
    s->launches += launchExclusiveScan(st, w.incPtr.p, n + 2, w.scanScratch.p);
    s->launches += launchSortPairs(st, nInc, w.incKeys.p, w.incVals.p, w.incTmpKeys.p, w.incTmpVals.p, w.sortHist.p, bitsFor(n));
    k_pbd_tickets<<<gridFor(nInc, kThreads), kThreads, 0, st>>>(nInc, w.incKeys.p, w.incVals.p, w.incPtr.p,
                                                               reinterpret_cast<uint32_t*>(w.visTk.p)); ++s->launches;
    if (w.countersUsed == 64) { PCHECK(cudaMemsetAsync(w.counters.p, 0, 64 * sizeof(uint32_t), st)); w.countersUsed = 0; }
    PCHECK(cudaMemsetAsync(w.nodeDone.p, 0, (size_t)(n + 2) * sizeof(uint32_t), st));
    uint32_t chunks = (nVis + 31u) / 32u;
    int grid = (int)std::min<uint32_t>(kNumSMs * 4, (chunks + kSweepThreads / 32 - 1) / (kSweepThreads / 32));
    k_pbd_collide<<<grid, kSweepThreads, 0, st>>>(nVis, w.visits.p, w.visTk.p, s->q.p, s->prev.p, w.turnStart.p, scale, kp,
                                                 w.q0.p, delta, w.flags.p, w.nodeDone.p, w.counters.p + w.countersUsed); ++s->launches;
    ++w.countersUsed;
    PCHECK(cudaMemcpyAsync(w.host + 11, w.flags.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    PCHECK(cudaStreamSynchronize(st));
    w.visitsLastTick += nVis;
    if (getenv("PIES_DEBUG_PBD"))
      std::fprintf(stderr, "[pbd] pairs %llu cells %u visits %u delta %g attempt %d -> %s\n", (unsigned long long)nPairs, nCells,
                   nVis, delta, attempt, w.host[11] ? "redo" : "ok");
    if (!w.host[11]) return PIES_B200_OK;
    // a node moved further than the pruning assumed: restore and redo with twice the bound
    PCHECK(cudaMemcpyAsync(s->q.p, w.q0.p, (size_t)n * sizeof(float4), cudaMemcpyDeviceToDevice, st));
    PCHECK(cudaMemsetAsync(w.flags.p, 0, sizeof(uint32_t), st));
    w.delta *= 2.0f;
  }
  s->simFailed = true;
  return fail(s, PIES_B200_ERANGE, "PBD node-node sweep: displacement bound not met after 8 attempts");
}

int tickPBD(PiesB200Solver* s, bool refreshMirror) {
  int rc = ensureBuilt(s);
  if (rc) return rc;
  const uint32_t n = s->n;
  s->stats.substepsLastTick = 0; s->stats.projectionsLastTick = 0; s->stats.pcgIterationsLastTick = 0;
  s->stats.msLocal = s->stats.msGlobal = s->stats.msDetect = s->stats.msContact = s->stats.msOther = 0.0f;
  s->stats.msTetKernel = 0.0f; s->stats.tetKernelLaunches = 0;
  s->stats.triCollisions = s->stats.staticCollisions = 0;
  const uint64_t launches0 = s->launches;
  if (!n) return PIES_B200_OK;
  if (!s->scene.tetW.empty())
    // Constraint<4,TetrahedralConstraintProjection>::projectNodePositions treats the differential coordinates the
    // projection returns as world positions (Constraints.h:121-129, Constraints.cpp:124-127): NaN on the first tick
    // in the reference (SURVEY F5).  There is nothing to be equal to; refuse instead of reproducing garbage.
    return fail(s, PIES_B200_EINVAL, "tickPBD with tetrahedral constraints is undefined in the reference (SURVEY F5)");
  if (!s->pbd) s->pbd = new PbdWork();
  PbdWork& w = *s->pbd;
  if (w.builtVersion != s->scene.topologyVersion && (rc = buildPbd(s, w))) return rc;
  if ((rc = prepareForces(s))) return rc;
  cudaStream_t st = s->stream;
  const PiesB200Options& o = s->opt;
  const float dt = o.fixedTimestepSize / (float)o.timeSubsteps;
  if ((rc = ensureTickEvents(s))) return rc;
  cudaEvent_t tick0 = s->tickEv[0], tick1 = s->tickEv[1];  // solver-owned: an early return below leaks nothing
  cudaEventRecord(tick0, st);
  PCHECK(cudaMemsetAsync(w.counters.p, 0, 64 * sizeof(uint32_t), st));
  w.countersUsed = 0; w.visitsLastTick = 0;
  PosOp pos{w.posIds.p, w.posTk.p, w.posTargetW.p};
  DistOp dist{w.distIds.p, w.distTk.p, w.distRestW.p};
  BendOp bend{w.bendIds.p, w.bendTk.p, w.bendAngleW.p};
  const ForceSet forces = forceSet(s);
  for (uint32_t sub = 0; sub < o.timeSubsteps; ++sub) {
    s->launches += launchForces(st, n, forces, s->q.p, s->vel.p);
    if (const float4* f = forces.field())
      k_pbd_advect<true><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, s->q.p, s->prev.p, s->vel.p, dt, o.gravity, f);
    else
      k_pbd_advect<false><<<gridFor(n, kThreads), kThreads, 0, st>>>(n, s->q.p, s->prev.p, s->vel.p, dt, o.gravity, nullptr);
    ++s->launches;
    for (uint32_t it = 0; it < o.iterations; ++it) {
      if (!s->releaseHinge && (rc = sweep(s, w, w.nPos, pos))) goto done;
      s->launches += launchPbdDrag(st, dragSet(s), s->q.p);
      if ((rc = sweep(s, w, w.nDist, dist))) goto done;
      if ((rc = sweep(s, w, w.nBend, bend))) goto done;
      if ((rc = collideNodes(s, w))) goto done;
      k_pbd_floor<<<gridFor(n, kThreads), kThreads, 0, st>>>(n, s->q.p, s->prev.p, o.floorHeight); ++s->launches;
      s->launches += launchPbdColliderClamp(st, n, colliderSet(s), s->q.p, s->prev.p);
      s->stats.projectionsLastTick += (s->releaseHinge ? 0u : w.nPos) + w.nDist + w.nBend;
    }
    k_pbd_velocity<<<gridFor(n, kThreads), kThreads, 0, st>>>(n, s->q.p, s->prev.p, s->vel.p, dt, o.damping, o.friction,
                                                             o.floorHeight); ++s->launches;
    s->launches += launchPbdColliderFriction(st, n, colliderSet(s), s->q.p, s->prev.p, s->vel.p, o.friction);
    ++s->stats.substepsLastTick;
  }
  s->stats.projectionsLastTick += w.visitsLastTick;
  s->stats.collisionProjections = w.visitsLastTick;
done:
  s->deviceNewer = true;
  cudaEventRecord(tick1, st);
  cudaError_t es = cudaEventSynchronize(tick1);
  cudaEventElapsedTime(&s->stats.msTick, tick0, tick1);
  if (rc) return rc;
  if (es != cudaSuccess) return failCuda(s, es, "cudaEventSynchronize", __LINE__);
  PCHECK(cudaGetLastError());
  s->mirrorStale = true;
  if (refreshMirror && (rc = refreshVertexMirror(s))) return rc;
  s->stats.kernelLaunchesLastTick = s->launches - launches0;
  s->stats.simFailed = s->simFailed ? 1u : 0u;
  return PIES_B200_OK;
}

// Runs only the node-hash build on the current state (parity tests; the PBD analogue of pies_b200_detect).
int pbdHashOnly(PiesB200Solver* s) {
  int rc = ensureBuilt(s);
  if (rc) return rc;
  if (!s->n) return PIES_B200_OK;
  if (!s->pbd) s->pbd = new PbdWork();
  PbdWork& w = *s->pbd;
  if (w.builtVersion != s->scene.topologyVersion && (rc = buildPbd(s, w))) return rc;
  NodeKeyPack kp{};
  return buildNodeHash(s, w, kp);
}

// Node-hash occupancy of the last PBD iteration, for the parity tests (cells sorted by (x,y,z), members ascending).
int pbdOccupancyCounts(PiesB200Solver* s, uint64_t* nCells, uint64_t* nMembers) {
  *nCells = s->pbd ? s->pbd->nCells : 0; *nMembers = s->pbd ? s->pbd->nPairs : 0;
  return PIES_B200_OK;
}

int pbdOccupancy(PiesB200Solver* s, int64_t* cellsXYZ, uint32_t* counts, uint32_t* members) {
  if (!s->pbd || !s->pbd->nPairs) return PIES_B200_OK;
  PbdWork& w = *s->pbd;
  std::vector<uint64_t> keys(w.nCells);
  std::vector<uint32_t> start(w.nCells + 1);
  PCHECK(cudaMemcpy(keys.data(), w.cellKey.p, w.nCells * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  PCHECK(cudaMemcpy(start.data(), w.cellStart.p, (w.nCells + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  PCHECK(cudaMemcpy(members, w.vals.p, w.nPairs * sizeof(uint32_t), cudaMemcpyDeviceToHost));
  const int by = w.keyPack[3], bz = w.keyPack[4];
  for (uint32_t c = 0; c < w.nCells; ++c) {
    uint64_t k = keys[c];
    cellsXYZ[3 * c + 2] = (int64_t)(k & ((1ull << bz) - 1ull)) + w.keyPack[2];
    cellsXYZ[3 * c + 1] = (int64_t)((k >> bz) & ((1ull << by) - 1ull)) + w.keyPack[1];
    cellsXYZ[3 * c + 0] = (int64_t)(k >> (by + bz)) + w.keyPack[0];
    counts[c] = start[c + 1] - start[c];
  }
  return PIES_B200_OK;
}

}  // namespace pies
