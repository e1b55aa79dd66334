// islands.cu — the global step of Projective Dynamics solved island by island.
//
// The reference factorises S + C_t as one sparse matrix every substep and solves with it (reference
// Src/Solver.cpp:242-262 SimplicialLLT(S + C_t), :356 solve).  That matrix is block diagonal: S couples only the nodes
// of one body, and the collision terms C_t (CollisionConstraint.cpp:74-83) couple bodies only where a point-triangle
// contact joins them.  A connected component of its graph — an "island": static bodies united through this substep's
// contacts — is an independent linear system, and nearly all of them are small (a free body; a column of stacked
// boxes).  So instead of a grid-wide CG whose every iteration streams the whole matrix from HBM and synchronises the
// device twice, every island is solved by its own team and stops on its own residual:  ||r_island|| <= tol ||b_island||
// per coordinate column (a stricter test than the same bound on the global norms).  An island that is one
// preconditioner block is refined by one warp with its exact block inverse, a small one by one CTA with its dense
// inverse; the CG team is one CTA that keeps the island's matrix, the inverses of its preconditioner blocks and the CG
// vectors in shared memory for the whole solve and iterates with CTA barriers only.  Only islands too large for one CTA
// go to the grid-wide CG (pcg.cu).
//
// Determinism: the island order (bodies ascending inside an island, nodes ascending inside a body) comes from a
// stable sort, every dot product is reduced in a fixed order inside the team, no float atomics.
#include "islands.h"

#include <algorithm>
#include <cstdlib>

#include "common.cuh"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ------------------------------------------------------------------------------------------------ builder ----
__device__ __forceinline__ uint32_t islFind(uint32_t* parent, uint32_t x) {
  uint32_t p = *(volatile uint32_t*)(parent + x);
  while (p != x) { x = p; p = *(volatile uint32_t*)(parent + x); }
  return x;
}
__device__ __forceinline__ void islUnite(uint32_t* parent, uint32_t u, uint32_t v) {
  while (true) {
    u = islFind(parent, u);
    v = islFind(parent, v);
    if (u == v) return;
    if (u < v) { uint32_t t = u; u = v; v = t; }  // hook the larger root under the smaller one
    uint32_t old = atomicMin(parent + u, v);
    if (old == u) return;
    u = old;
  }
}

__global__ void __launch_bounds__(kThreads) k_isl_init(uint32_t nB, uint32_t* __restrict__ parent) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < nB) parent[b] = b;
}

__global__ void __launch_bounds__(kThreads) k_isl_unite(uint32_t nU, const uint4* __restrict__ uTri,
                                                        const uint32_t* __restrict__ bodyOf, uint32_t* __restrict__ parent) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nU) return;
  const uint4 id = uTri[e];
  const uint32_t a = bodyOf[id.x], b = bodyOf[id.y], c = bodyOf[id.z], d = bodyOf[id.w];
  if (a != b) islUnite(parent, a, b);
  if (c != b) islUnite(parent, b, c);
  if (d != b && d != c) islUnite(parent, b, d);
}

// sort keys: the island's root body; payload: the body.  Without contacts every body is its own island.
__global__ void __launch_bounds__(kThreads) k_isl_keys(uint32_t nB, uint32_t* __restrict__ parent, int united,
                                                       uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nB) return;
  keys[b] = united ? islFind(parent, b) : b;
  vals[b] = b;
}

// per sorted body: head flag (to be scanned into the island index) and node count (to be scanned into node offsets)
__global__ void __launch_bounds__(kThreads) k_isl_heads(uint32_t nB, const uint64_t* __restrict__ keys,
                                                        const uint32_t* __restrict__ vals, const uint32_t* __restrict__ bodyPtr,
                                                        uint32_t* __restrict__ heads, uint32_t* __restrict__ nodeOff,
                                                        uint32_t* __restrict__ posOfBody) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > nB) return;
  if (j == nB) { heads[j] = 0; nodeOff[j] = 0; return; }
  heads[j] = (j == 0 || keys[j] != keys[j - 1]) ? 1u : 0u;
  const uint32_t b = vals[j];
  nodeOff[j] = bodyPtr[b + 1] - bodyPtr[b];
  posOfBody[b] = j;
}

__global__ void __launch_bounds__(kThreads) k_isl_starts(uint32_t nB, uint32_t n, const uint64_t* __restrict__ keys,
                                                         const uint32_t* __restrict__ headScan,
                                                         const uint32_t* __restrict__ nodeOff, uint32_t* __restrict__ islStart,
                                                         uint32_t* __restrict__ counts) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nB) return;
  const bool head = j == 0 || keys[j] != keys[j - 1];
  if (head) islStart[headScan[j]] = nodeOff[j];
  if (j == nB - 1) {
    const uint32_t nIsl = headScan[nB];
    islStart[nIsl] = n;
    counts[0] = nIsl;
  }
}

// island order of the nodes, its inverse, and the row lengths of S + C_t in that order (to be scanned)
__global__ void __launch_bounds__(kThreads) k_isl_nodes(uint32_t n, const uint32_t* __restrict__ bodyOf,
                                                        const uint32_t* __restrict__ rankInBody,
                                                        const uint32_t* __restrict__ posOfBody,
                                                        const uint32_t* __restrict__ nodeOff, const int* __restrict__ rowPtr,
                                                        const int* __restrict__ cPtr, uint32_t* __restrict__ order,
                                                        uint32_t* __restrict__ pos, uint32_t* __restrict__ nnzOff) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { nnzOff[n] = 0; return; }
  const uint32_t p = nodeOff[posOfBody[bodyOf[i]]] + rankInBody[i];
  order[p] = i;
  pos[i] = p;
  uint32_t len = (uint32_t)(rowPtr[i + 1] - rowPtr[i]);
  if (cPtr) len += (uint32_t)(cPtr[i + 1] - cPtr[i]);
  nnzOff[p] = len;
}

// ------------------------------------------------------------------------------------------------- lists -----
// An island goes to the first list of kClassifyOrder whose public tier is on and whose caps it fits, or to the grid-wide
// CG (device list kIslandLists).  The public tier is the islandsTier entry of PiesB200Stats and the tuning bit 16 << tier.
enum IslandKind : int { kDirect, kDense, kCtaCg, kBig };   // k_island_direct / _invert + _dense / _pcg / _pcg_big
constexpr uint32_t kDenseMax = 128;   // node caps of the dense lists; the inverse is stored with this leading dimension
constexpr uint32_t kDenseMax2 = 192;
struct IslandCaps { uint32_t maxNodes, maxNnz, maxInv, maxBlocks; };
// A/B switches that take lists out (environment, read once per process): PIES_B200_NO_SMALL_CTA, _NO_DENSE, _NO_DENSE2
constexpr uint32_t kNoSmallCta = 1, kNoDense = 2, kNoDense2 = 4;
struct IslandList {
  IslandKind kind;      // also which inverse a solve reads: the packed block inverse, the dense one, the blocks' ones
  int team, rpt;        // threads of the team solving one island, rows per thread
  IslandCaps caps;      // nodes, matrix entries, inverse floats, blocks resident in shared memory
  int tier;             // public tier
  int ctasPerSm;        // grid cap of a solve
  int shortList;        // a list that fits one wave of this list's CTAs goes to its team: a short list is latency bound
  uint32_t offBy;       // A/B switches
};
constexpr IslandList kLists[kIslandLists] = {
    {kDirect, 32, 1, {32u, 640u, 576u, 4u}, 0, 4, 0, 0u},            // 0: every free body; eight warps per CTA
    {kCtaCg, 320, 2, {640u, 6656u, 9216u, 96u}, 1, 2, 1, 0u},
    {kCtaCg, 512, 2, {1024u, 12288u, 17408u, 192u}, 2, 1, 2, 0u},   // 2: the whole shared memory of an SM
    {kBig, 1024, 0, {7168u, 0u, 0u, 0u}, 3, 1, 3, 0u},               // 3: opt-in
    // 4: the typical S3 contact island is five bodies (~140 rows), which leaves more than half of a 320-thread CTA
    //    waiting at every barrier: 43 KB of shared memory, five CTAs per SM
    {kCtaCg, 128, 2, {256u, 2816u, 3456u, 32u}, 1, 5, 1, kNoSmallCta},
    {kDense, (int)kDenseMax, 1, {kDenseMax, 0u, 0u, 0u}, 1, 16, 5, kNoDense},                 // 5: 3-4 bodies of a column
    // 6: 5-7 bodies (S3 ticks 79..100); beyond that the m^3 of the inversion and the m^2 of every apply lose to the CG
    {kDense, (int)kDenseMax2, 1, {kDenseMax2, 0u, 0u, 0u}, 1, 10, 6, kNoDense | kNoDense2},
};
constexpr int kClassifyOrder[kIslandLists] = {0, 5, 6, 4, 1, 2, 3};   // cheapest solve first
constexpr int kLaunchOrder[kIslandLists] = {3, 2, 1, 4, 6, 5, 0};     // longest chains first

// the lists in classification order, with their numbers, as the A/B switches and the tuning word leave them
struct IslandClassifyTable { IslandList list[kIslandLists]; int id[kIslandLists]; uint32_t tiersOn; };

__global__ void __launch_bounds__(kThreads) k_isl_classify(const uint32_t* counts0, IslandClassifyTable tt,
                                                           const uint32_t* __restrict__ islStart,
                                                           const uint32_t* __restrict__ nnzOff, const uint32_t* __restrict__ order,
                                                           const uint32_t* __restrict__ slotOf,
                                                           const uint32_t* __restrict__ blockCount, uint32_t listStride,
                                                           uint32_t* __restrict__ tierList, uint4* __restrict__ tierDesc,
                                                           uint32_t* counts) {
  uint32_t isl = blockIdx.x * blockDim.x + threadIdx.x;
  if (isl >= counts0[0]) return;
  const uint32_t s0 = islStart[isl], m = islStart[isl + 1] - s0;
  const uint32_t nnz = nnzOff[s0 + m] - nnzOff[s0];
  int list = kIslandLists;
  IslandKind kind = kCtaCg;
#pragma unroll
  for (int o = 0; o < kIslandLists; ++o) {
    const IslandList& e = tt.list[o];
    if (!((tt.tiersOn >> e.tier) & 1u)) continue;
    if (m > e.caps.maxNodes || (e.caps.maxNnz && nnz > e.caps.maxNnz)) continue;
    if (e.kind == kDirect && blockCount[slotOf[order[s0]] >> 5] != m) continue;  // the island must be ONE preconditioner block
    list = tt.id[o];
    kind = e.kind;
    break;
  }
  const uint32_t at = atomicAdd(counts + 1 + list, 1u);  // list order only decides scheduling: islands are independent
  tierList[(size_t)list * listStride + at] = isl;
  // everything a team needs to start on the island in one 16 B record (it prefetches the next one while it solves)
  tierDesc[(size_t)list * listStride + at] = make_uint4(isl, s0, m, nnzOff[s0]);
  if (list == kIslandLists) atomicAdd(counts + 2 + kIslandLists, m);
  // floats of inverse the island's solve has to read (CG lists: at most 16.5 per node, taken as 14 = a 27-node block)
  else atomicAdd(counts + 3 + kIslandLists, kind == kDirect ? m * (m + 1u) / 2u : (kind == kDense ? m * m : 14u * m));
}

// Marks the nodes of the islands left to the grid-wide CG, the 256-row windows that hold one and their preconditioner
// blocks (one CTA per left-over island; they are few and large).
__global__ void __launch_bounds__(kThreads) k_isl_mark_big(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ list,
                                                           const uint32_t* __restrict__ islStart, const uint32_t* __restrict__ order,
                                                           const uint32_t* __restrict__ slotOf, uint8_t* __restrict__ big,
                                                           uint32_t* __restrict__ winFlag, uint32_t* __restrict__ blkFlag) {
  const uint32_t nLeft = counts[1 + kIslandLists];
  for (uint32_t k = blockIdx.x; k < nLeft; k += gridDim.x) {
    const uint32_t isl = list[k];
    const uint32_t s0 = islStart[isl], m = islStart[isl + 1] - s0;
    for (uint32_t l = threadIdx.x; l < m; l += blockDim.x) {
      const uint32_t g = order[s0 + l];
      big[g] = 1;
      winFlag[g >> 8] = 1u;            // benign race: every writer stores 1
      blkFlag[slotOf[g] >> 5] = 1u;
    }
  }
}

// ascending list of the set flags from their exclusive scan; the count goes to out count
__global__ void __launch_bounds__(kThreads) k_isl_compact(uint32_t n, const uint32_t* __restrict__ scan, uint32_t* __restrict__ list,
                                                          uint32_t* __restrict__ count) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { *count = scan[n]; return; }
  if (scan[i + 1] != scan[i]) list[scan[i]] = i;
}

// ------------------------------------------------------------------------------------------------ solver ----
struct IslandLayout { uint32_t r, p, val, inv, blkOff, blkSrc, col, members, leader, blkM, red, ctr, total; };

static IslandLayout islandLayout(const IslandCaps& c) {
  IslandLayout L{};
  uint32_t off = 0;
  auto take = [&](uint32_t bytes) { uint32_t at = off; off += (bytes + 15u) & ~15u; return at; };
  L.r = take(16u * c.maxNodes);
  L.p = take(16u * c.maxNodes);
  L.val = take(4u * c.maxNnz);
  L.inv = take(4u * c.maxInv);
  L.blkOff = take(4u * c.maxBlocks);
  L.blkSrc = take(4u * c.maxBlocks);
  L.col = take(2u * c.maxNnz);
  L.members = take(64u * c.maxBlocks);
  L.leader = take(c.maxBlocks ? 2u * c.maxNodes : 0u);
  L.blkM = take(c.maxBlocks);
  L.red = take(2u * 9u * 32u * 4u);
  L.ctr = take(16u);
  L.total = off;
  return L;
}

struct IslandArgs {
  const uint32_t* counts; const uint32_t* tierList; const uint4* tierDesc; uint32_t listStride;
  const uint32_t* islStart; const uint32_t* order; const uint32_t* pos; const uint32_t* nnzOff;
  const int* rowPtr; const int* col; const float* val; const uint32_t* colRank; const uint32_t* rankInBody;
  const int* cPtr; const int* cCol; const float* cVal; const float* cDiag;
  const uint32_t* slotOf; const int* blockNodes; const float* blockInv; const uint2* blockMeta;
  uint32_t* blkLocal;          // block * 32 + lane -> local row of that member (scratch, written per solve)
  int* matCol; float* matVal;  // tier 3 scratch copy of the matrix in island-local indices
  float4* deltaScratch;        // tier 3: accumulated correction, island order
  float4* apScratch; float4* zScratch; uint32_t* slotIsl;  // tier 3: A p, z and the preconditioner slot per row, island order
  const float4* b; float4* x;
  float tol2; uint32_t maxIter; uint32_t* stats;
  uint4* trace;                // diagnostics: per list entry (rows, iterations, clocks, matrix entries), or null
};

// Fixed-order sum of K values per thread over the CTA; every thread gets the result.  The CTA alternates between two
// scratch buffers, so one barrier per reduction is enough.
template <int TEAM, int K>
__device__ __forceinline__ void teamReduce(float (&v)[K], float* __restrict__ sRed, int& phase, int tid) {
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = warpSum(v[k]);
  float* buf = sRed + phase * (9 * 32);
  phase ^= 1;
  const int lane = tid & 31, warp = tid >> 5;
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) buf[k * 32 + warp] = v[k];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < K; ++k) {
    const float t = lane < TEAM / 32 ? buf[k * 32 + lane] : 0.0f;
    v[k] = warpSum(t);
  }
}

// The three-column convergence test of every island solve: ||r|| <= tol ||b|| per coordinate column, squared.
__device__ __forceinline__ bool converged3(const float (&rr)[3], const float (&bb)[3], float tol2) {
  return rr[0] <= tol2 * bb[0] + 1e-36f && rr[1] <= tol2 * bb[1] + 1e-36f && rr[2] <= tol2 * bb[2] + 1e-36f;
}

// One island's entry in its solve's 4-word statistics record (IslandWork::solveStats, read by the host once per tick):
// max iterations, iterations x 32-row units, islands stopped at the cap and their worst relative residual.
__device__ __forceinline__ void recordSolve(uint32_t* stats, uint32_t iters, uint32_t m, bool conv, const float (&rr)[3],
                                            const float (&bb)[3]) {
  atomicMax(stats, iters);
  atomicAdd(stats + 1, iters * ((m + 31u) >> 5));
  if (!conv) {
    float rel = 0.0f;
    for (int c = 0; c < 3; ++c) if (bb[c] > 0.0f) rel = fmaxf(rel, rr[c] / bb[c]);
    atomicAdd(stats + 2, 1u);
    atomicMax(stats + 3, __float_as_uint(sqrtf(rel)));
  }
}

// One CTA of TEAM threads per island, RPT rows per thread.
template <int TEAM, int RPT>
__global__ void __launch_bounds__(TEAM, TEAM <= 128 ? 5 : (TEAM <= 320 ? 2 : 1)) k_island_pcg(IslandArgs a, IslandLayout L, IslandCaps caps, int tier) {
  extern __shared__ __align__(16) unsigned char islSmem[];
  const int tid = (int)threadIdx.x;
  float4* sR = reinterpret_cast<float4*>(islSmem + L.r);
  float4* sP = reinterpret_cast<float4*>(islSmem + L.p);
  float* sInv = reinterpret_cast<float*>(islSmem + L.inv);
  uint32_t* sBlkOff = reinterpret_cast<uint32_t*>(islSmem + L.blkOff);
  uint32_t* sBlkSrc = reinterpret_cast<uint32_t*>(islSmem + L.blkSrc);
  uint16_t* sMem = reinterpret_cast<uint16_t*>(islSmem + L.members);
  uint16_t* sLeader = reinterpret_cast<uint16_t*>(islSmem + L.leader);
  uint8_t* sBlkM = reinterpret_cast<uint8_t*>(islSmem + L.blkM);
  float* sRed = reinterpret_cast<float*>(islSmem + L.red);
  uint32_t* sCtr = reinterpret_cast<uint32_t*>(islSmem + L.ctr);
  const uint32_t count = a.counts[1 + tier];
  const uint4* descs = a.tierDesc + (size_t)tier * a.listStride;
  int phase = 0;
  const uint32_t stride = gridDim.x;
  uint32_t wi = blockIdx.x;
  uint4 descNext = wi < count ? __ldg(descs + wi) : make_uint4(0u, 0u, 0u, 0u);
  for (; wi < count; wi += stride) {
    const uint4 desc = descNext;
    if (wi + stride < count) descNext = __ldg(descs + wi + stride);  // in flight while this island is solved
    const uint32_t s0 = desc.y, m = desc.z, z0 = desc.w;
    const long long t0 = a.trace ? clock64() : 0ll;
    float* mv = reinterpret_cast<float*>(islSmem + L.val);
    uint16_t* mc = reinterpret_cast<uint16_t*>(islSmem + L.col);
    if (tid == 0) { sCtr[0] = 0; sCtr[1] = 0; }
    __syncthreads();
    // ---- stage the island.  Rows are re-indexed without a gather per entry: S never leaves a body and the island order
    //      keeps a body's nodes together by rank, so local column = (row's body base) + rank of the column (host table).
    //      x of the island goes to sP and b to sR for the start residual below.
    uint32_t rs[RPT], rn[RPT], rb[RPT], slot[RPT], gid[RPT];
    float dl[RPT][3], cdg[RPT];
    float red9[9] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};  // r.z (3), r.r (3), b.b (3)
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
      rs[k] = 0; rn[k] = 0; rb[k] = 0xffffffffu; slot[k] = 0; gid[k] = 0; cdg[k] = 0.0f;
      dl[k][0] = dl[k][1] = dl[k][2] = 0.0f;
      if (l >= m) continue;
      const uint32_t g = a.order[s0 + l];
      gid[k] = g;
      const uint32_t rstart = a.nnzOff[s0 + l] - z0, rend = a.nnzOff[s0 + l + 1] - z0;
      rs[k] = rstart; rn[k] = rend - rstart;
      const int kk0 = a.rowPtr[g], kk1 = a.rowPtr[g + 1];
      const uint32_t bodyBase = l - a.rankInBody[g];
      const float4 bi = a.b[g];
      sP[l] = a.x[g]; sR[l] = bi;
      cdg[k] = a.cDiag ? a.cDiag[g] : 0.0f;
      const uint32_t sl = a.slotOf[g];
      slot[k] = sl;
      // (putting the loads of eight entries in flight together helped the staged warp tier, r02g: 85 -> 75 us; on a
      // CTA it costs registers and 10 %)
      uint32_t e = rstart;
#pragma unroll 4
      for (int kk = kk0; kk < kk1; ++kk) {
        const uint32_t rk = __ldg(a.colRank + kk);
        const float v = __ldg(a.val + kk);
        const bool out = rk == 0xffffffffu;  // an explicit zero pointing outside the body (bend stencils): dropped
        mc[e + (kk - kk0)] = (uint16_t)(out ? l : bodyBase + rk);
        mv[e + (kk - kk0)] = out ? 0.0f : v;
      }
      e += (uint32_t)(kk1 - kk0);
      if (a.cPtr) {
        const int c0 = a.cPtr[g], c1 = a.cPtr[g + 1];
        for (int kk = c0; kk < c1; ++kk) {
          mc[e + (kk - c0)] = (uint16_t)(__ldg(a.pos + __ldg(a.cCol + kk)) - s0);
          mv[e + (kk - c0)] = __ldg(a.cVal + kk);
        }
      }
      red9[6] += bi.x * bi.x; red9[7] += bi.y * bi.y; red9[8] += bi.z * bi.z;
      a.blkLocal[sl] = l;
      if (caps.maxBlocks) {
        sLeader[l] = 0xffffu;
        if ((sl & 31u) == 0u) {  // first member of its block: claim a table entry and room for the inverse
          const uint2 meta = __ldg(a.blockMeta + (sl >> 5));
          const uint32_t size = (meta.y * (meta.y + 1u) / 2u + 3u) & ~3u;
          const uint32_t idx = atomicAdd(sCtr, 1u);
          if (idx < caps.maxBlocks) {
            const uint32_t off = atomicAdd(sCtr + 1, size);
            if (off + size <= caps.maxInv) { sBlkOff[idx] = off; sBlkSrc[idx] = meta.x; sBlkM[idx] = (uint8_t)meta.y; sLeader[l] = (uint16_t)idx; }
            else sBlkM[idx] = 0;
          }
        }
      }
    }
    __syncthreads();
    // start residual r = b - A x from shared memory, accumulated in fp64 (float products are exact in double): b and A x
    // agree to ~7 digits and the difference is what matters
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
      if (l >= m) continue;
      const float4 xi = sP[l];
      double y0 = (double)cdg[k] * (double)xi.x, y1 = (double)cdg[k] * (double)xi.y, y2 = (double)cdg[k] * (double)xi.z;
      const uint32_t e1 = rs[k] + rn[k];
#pragma unroll 4
      for (uint32_t e = rs[k]; e < e1; ++e) {
        const double v = (double)mv[e];
        const float4 xv = sP[mc[e]];
        y0 += v * (double)xv.x; y1 += v * (double)xv.y; y2 += v * (double)xv.z;
      }
      const float4 bi = sR[l];
      sR[l] = make_float4((float)((double)bi.x - y0), (float)((double)bi.y - y1), (float)((double)bi.z - y2), 0.0f);
    }
    __syncthreads();
    if (caps.maxBlocks) {
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
        if (l >= m) continue;
        const uint32_t lead = a.pos[a.blockNodes[(slot[k] >> 5) * 32]] - s0;
        const uint32_t idx = sLeader[lead];
        if (idx != 0xffffu) { rb[k] = (idx << 5) | (slot[k] & 31u); sMem[idx * 32 + (slot[k] & 31u)] = (uint16_t)l; }
      }
      __syncthreads();
      // inverses: one warp per block, 16 B per lane and step
      const uint32_t nBlk = min(sCtr[0], caps.maxBlocks);
      for (uint32_t idx = (uint32_t)tid >> 5; idx < nBlk; idx += TEAM / 32) {
        const uint32_t mB = sBlkM[idx];
        if (!mB) continue;
        const uint32_t size4 = (mB * (mB + 1u) / 2u + 3u) >> 2;
        const float4* src = reinterpret_cast<const float4*>(a.blockInv + sBlkSrc[idx]);
        float4* dst = reinterpret_cast<float4*>(sInv + sBlkOff[idx]);
        for (uint32_t t = (uint32_t)tid & 31u; t < size4; t += 32u) dst[t] = __ldg(src + t);
      }
    }
    __syncthreads();

    // z = Minv r for one of this thread's rows
    auto precond = [&](int k, float (&z)[3]) {
      z[0] = z[1] = z[2] = 0.0f;
      if (rb[k] != 0xffffffffu) {
        const uint32_t idx = rb[k] >> 5;
        const int lane = (int)(rb[k] & 31u), mB = (int)sBlkM[idx];
        const float* inv = sInv + sBlkOff[idx];
        const uint16_t* mem = sMem + idx * 32;
        int off = lane * (lane + 1) / 2;
#pragma unroll 3
        for (int j = 0; j < mB; ++j) {
          const float w = inv[off];
          const float4 rj = sR[mem[j]];
          z[0] = fmaf(w, rj.x, z[0]); z[1] = fmaf(w, rj.y, z[1]); z[2] = fmaf(w, rj.z, z[2]);
          off += j < lane ? 1 : j + 1;
        }
      } else {  // block not resident (the island has more blocks than the tier's table): same sum from global memory
        const uint32_t b = slot[k] >> 5;
        const int lane = (int)(slot[k] & 31u);
        const uint2 meta = a.blockMeta[b];
        const float* inv = a.blockInv + meta.x;
        const uint32_t* loc = a.blkLocal + (size_t)b * 32;
        const int tri = lane * (lane + 1) / 2;
        for (int j = 0; j < (int)meta.y; ++j) {
          const float w = __ldg(inv + (j < lane ? tri + j : j * (j + 1) / 2 + lane));
          const float4 rj = sR[loc[j]];
          z[0] = fmaf(w, rj.x, z[0]); z[1] = fmaf(w, rj.y, z[1]); z[2] = fmaf(w, rj.z, z[2]);
        }
      }
    };

    // ---- CG on the correction delta (x is updated once at the end: a single rounding of the sum).  Plain two-reduction
    //      CG: the single-reduction (Chronopoulos-Gear) arrangement was measured too (r02c): 4 % faster on the CTA tier,
    //      slower on the warp tier (one extra preconditioner + mat-vec per solve), and its recurrences cost accuracy.
    float zz[RPT][3];
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
      if (l >= m) continue;
      precond(k, zz[k]);
      const float4 r = sR[l];
      red9[0] += r.x * zz[k][0]; red9[1] += r.y * zz[k][1]; red9[2] += r.z * zz[k][2];
      red9[3] += r.x * r.x; red9[4] += r.y * r.y; red9[5] += r.z * r.z;
      sP[l] = make_float4(zz[k][0], zz[k][1], zz[k][2], 0.0f);
    }
    teamReduce<TEAM, 9>(red9, sRed, phase, tid);
    float rz[3] = {red9[0], red9[1], red9[2]};
    float rr[3] = {red9[3], red9[4], red9[5]};
    const float bb[3] = {red9[6], red9[7], red9[8]};
    __syncthreads();  // p visible
    uint32_t iters = 0;
    bool conv = converged3(rr, bb, a.tol2);
    while (!conv && iters < a.maxIter) {
      float ap[RPT][3];
      float pap[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
        ap[k][0] = ap[k][1] = ap[k][2] = 0.0f;
        if (l >= m) continue;
        const uint32_t e1 = rs[k] + rn[k];
#pragma unroll 4
        for (uint32_t e = rs[k]; e < e1; ++e) {
          const float v = mv[e];
          const float4 pv = sP[mc[e]];
          ap[k][0] = fmaf(v, pv.x, ap[k][0]); ap[k][1] = fmaf(v, pv.y, ap[k][1]); ap[k][2] = fmaf(v, pv.z, ap[k][2]);
        }
        const float4 pl = sP[l];
        ap[k][0] = fmaf(cdg[k], pl.x, ap[k][0]); ap[k][1] = fmaf(cdg[k], pl.y, ap[k][1]); ap[k][2] = fmaf(cdg[k], pl.z, ap[k][2]);
        pap[0] += pl.x * ap[k][0]; pap[1] += pl.y * ap[k][1]; pap[2] += pl.z * ap[k][2];
      }
      teamReduce<TEAM, 3>(pap, sRed, phase, tid);
      float alpha[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) alpha[c] = pap[c] > 0.0f ? rz[c] / pap[c] : 0.0f;
      float rl[RPT][3];
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
        if (l >= m) continue;
        const float4 pl = sP[l];
        dl[k][0] = fmaf(alpha[0], pl.x, dl[k][0]); dl[k][1] = fmaf(alpha[1], pl.y, dl[k][1]); dl[k][2] = fmaf(alpha[2], pl.z, dl[k][2]);
        const float4 r = sR[l];
        rl[k][0] = fmaf(-alpha[0], ap[k][0], r.x); rl[k][1] = fmaf(-alpha[1], ap[k][1], r.y); rl[k][2] = fmaf(-alpha[2], ap[k][2], r.z);
        sR[l] = make_float4(rl[k][0], rl[k][1], rl[k][2], 0.0f);
      }
      __syncthreads();  // r visible
      float red6[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
        if (l >= m) continue;
        precond(k, zz[k]);
        red6[0] += rl[k][0] * zz[k][0]; red6[1] += rl[k][1] * zz[k][1]; red6[2] += rl[k][2] * zz[k][2];
        red6[3] += rl[k][0] * rl[k][0]; red6[4] += rl[k][1] * rl[k][1]; red6[5] += rl[k][2] * rl[k][2];
      }
      teamReduce<TEAM, 6>(red6, sRed, phase, tid);
      float beta[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) { beta[c] = rz[c] > 0.0f ? red6[c] / rz[c] : 0.0f; rz[c] = red6[c]; rr[c] = red6[3 + c]; }
      ++iters;
      conv = converged3(rr, bb, a.tol2);
      if (conv) break;
#pragma unroll
      for (int k = 0; k < RPT; ++k) {
        const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
        if (l >= m) continue;
        const float4 pl = sP[l];
        sP[l] = make_float4(fmaf(beta[0], pl.x, zz[k][0]), fmaf(beta[1], pl.y, zz[k][1]), fmaf(beta[2], pl.z, zz[k][2]), 0.0f);
      }
      __syncthreads();  // p visible
    }
#pragma unroll
    for (int k = 0; k < RPT; ++k) {
      const uint32_t l = (uint32_t)tid + (uint32_t)k * TEAM;
      if (l >= m) continue;
      float4 xv = a.x[gid[k]];
      xv.x += dl[k][0]; xv.y += dl[k][1]; xv.z += dl[k][2];
      a.x[gid[k]] = xv;
    }
    if (tid == 0) {
      recordSolve(a.stats, iters, m, conv, rr, bb);
      if (a.trace)
        a.trace[(size_t)tier * a.listStride + wi] = make_uint4(m, iters, (uint32_t)(clock64() - t0), a.nnzOff[s0 + m] - z0);
    }
    __syncthreads();  // the CTA's shared memory is restaged for its next island
  }
}

// Tier 0 without staging: one warp per island that is a single preconditioner block (every free body of a multi-body
// scene).  The block inverse is then the exact inverse of the island's matrix (contact diagonal included: such blocks are
// re-inverted by reblock.cu), so the solve is iterative refinement rather than CG:  r = b - A x in fp64, z = Minv r,
// x += z, r -= A z, until the island's residual passes the tolerance (a round contracts the residual by ~1e-5).  The
// vectors live one row per lane and move by shuffles — every column of an island row lies in the island, so nothing is
// gathered from global memory — the matrix rows are read where they lie, the block's packed inverse travels to shared
// memory with cp.async while the start residual is computed, and with 64 registers four CTAs of eight warps fit an SM,
// which is what a kernel bound by dependent global loads needs (r02g: the staged warp tier was long-scoreboard bound at
// 24 warps per SM).
__global__ void __launch_bounds__(256, 4) k_island_direct(IslandArgs a, int tier) {
  __shared__ __align__(16) float sInv[8][528];   // the block's packed inverse (at most 32 * 33 / 2 floats), one per warp
  __shared__ unsigned char sLaneOf[8][32];
  const int lane = (int)(threadIdx.x & 31), warp = (int)(threadIdx.x >> 5);
  const uint32_t count = a.counts[1 + tier];
  const uint4* descs = a.tierDesc + (size_t)tier * a.listStride;
  const uint32_t stride = gridDim.x * 8u;
  uint32_t wi = blockIdx.x * 8u + (uint32_t)warp;
  uint4 descNext = wi < count ? __ldg(descs + wi) : make_uint4(0u, 0u, 0u, 0u);
  for (; wi < count; wi += stride) {
    const uint4 desc = descNext;
    if (wi + stride < count) descNext = __ldg(descs + wi + stride);
    const uint32_t s0 = desc.y, m = desc.z;
    const bool act = (uint32_t)lane < m;
    uint32_t g = 0, sl = 0, bodyBase = 0;
    int kk0 = 0, kk1 = 0, c0 = 0, c1 = 0;
    float4 xi = make_float4(0.0f, 0.0f, 0.0f, 0.0f), bi = xi;
    float cd = 0.0f;
    if (act) {
      g = a.order[s0 + lane];
      kk0 = a.rowPtr[g]; kk1 = a.rowPtr[g + 1];
      xi = a.x[g]; bi = a.b[g];
      cd = a.cDiag ? a.cDiag[g] : 0.0f;
      sl = a.slotOf[g];
      bodyBase = (uint32_t)lane - a.rankInBody[g];
      if (a.cPtr) { c0 = a.cPtr[g]; c1 = a.cPtr[g + 1]; }
    }
    const int bl = (int)(sl & 31u);
    // the block's inverse is indexed by block lane: which island lane holds block lane j
    __syncwarp();
    if (act) sLaneOf[warp][bl] = (unsigned char)lane;
    const uint32_t blk = __shfl_sync(0xffffffffu, sl, 0) >> 5;
    const uint2 meta = __ldg(a.blockMeta + blk);
    const int mB = (int)meta.y;
    {  // the inverse travels to shared memory asynchronously while the start residual is computed
      const uint32_t n4 = ((uint32_t)(mB * (mB + 1) / 2) + 3u) >> 2;
      const float4* src = reinterpret_cast<const float4*>(a.blockInv + meta.x);
      const uint32_t dst = (uint32_t)__cvta_generic_to_shared(&sInv[warp][0]);
      for (uint32_t t = (uint32_t)lane; t < n4; t += 32u)
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst + 16u * t), "l"(src + t) : "memory");
      asm volatile("cp.async.commit_group;\n" ::: "memory");
    }
    // ---- the row's entries as (value, island lane of the column): every column of an island row lies in the island, so
    //      vectors move by shuffles and nothing is gathered from global memory.  Entry k of the row: S entries through
    //      the host's rank table (an explicit zero pointing outside the body is dropped), then this substep's contacts.
    const int maxLen = __reduce_max_sync(0xffffffffu, (kk1 - kk0) + (c1 - c0));
    auto entry = [&](int k, float& v, int& src) {
      v = 0.0f; src = lane;
      const int ks = kk0 + k;
      if (ks < kk1) {
        const uint32_t rk = __ldg(a.colRank + ks);
        if (rk != 0xffffffffu) { v = __ldg(a.val + ks); src = (int)(bodyBase + rk); }
      } else if (c0 + (ks - kk1) < c1) {
        const int kc = c0 + (ks - kk1);
        v = a.cVal[kc]; src = (int)(__ldg(a.pos + a.cCol[kc]) - s0);
      }
    };
    // ---- start residual, fp64 accumulation
    double y0 = (double)cd * (double)xi.x, y1 = (double)cd * (double)xi.y, y2 = (double)cd * (double)xi.z;
    for (int k = 0; k < maxLen; k += 2) {   // two entries per step: their loads are in flight together
      float v[2]; int src[2];
      entry(k, v[0], src[0]);
      if (k + 1 < maxLen) entry(k + 1, v[1], src[1]); else { v[1] = 0.0f; src[1] = lane; }
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const float q0 = __shfl_sync(0xffffffffu, xi.x, src[u]), q1 = __shfl_sync(0xffffffffu, xi.y, src[u]), q2 = __shfl_sync(0xffffffffu, xi.z, src[u]);
        y0 += (double)v[u] * (double)q0; y1 += (double)v[u] * (double)q1; y2 += (double)v[u] * (double)q2;
      }
    }
    float r0 = 0.0f, r1 = 0.0f, r2 = 0.0f;
    if (act) { r0 = (float)((double)bi.x - y0); r1 = (float)((double)bi.y - y1); r2 = (float)((double)bi.z - y2); }
    const float bb[3] = {warpSum(bi.x * bi.x), warpSum(bi.y * bi.y), warpSum(bi.z * bi.z)};
    float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f;
    uint32_t iters = 0;
    bool conv = false;
    float rr[3];
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncwarp();
    const float* inv = &sInv[warp][0];
    while (true) {
      rr[0] = warpSum(r0 * r0); rr[1] = warpSum(r1 * r1); rr[2] = warpSum(r2 * r2);
      conv = converged3(rr, bb, a.tol2);
      if (conv || iters >= a.maxIter) break;
      // z = Minv r: lane with block lane bl owns row bl of the packed lower triangle
      float z0 = 0.0f, z1 = 0.0f, z2 = 0.0f;
      {
        int off = bl * (bl + 1) / 2;
#pragma unroll 4
        for (int j = 0; j < mB; ++j) {
          const float w = act ? inv[off] : 0.0f;
          const int src = (int)sLaneOf[warp][j];
          const float q0 = __shfl_sync(0xffffffffu, r0, src), q1 = __shfl_sync(0xffffffffu, r1, src), q2 = __shfl_sync(0xffffffffu, r2, src);
          z0 = fmaf(w, q0, z0); z1 = fmaf(w, q1, z1); z2 = fmaf(w, q2, z2);
          off += j < bl ? 1 : j + 1;
        }
      }
      d0 += z0; d1 += z1; d2 += z2;
      // r -= A z
      float w0 = cd * z0, w1 = cd * z1, w2 = cd * z2;
      for (int k = 0; k < maxLen; ++k) {
        float v; int src;
        entry(k, v, src);
        const float q0 = __shfl_sync(0xffffffffu, z0, src), q1 = __shfl_sync(0xffffffffu, z1, src), q2 = __shfl_sync(0xffffffffu, z2, src);
        w0 = fmaf(v, q0, w0); w1 = fmaf(v, q1, w1); w2 = fmaf(v, q2, w2);
      }
      r0 -= w0; r1 -= w1; r2 -= w2;
      ++iters;
    }
    if (act) {
      xi.x += d0; xi.y += d1; xi.z += d2;
      a.x[g] = xi;
    }
    if (lane == 0) {
      recordSolve(a.stats, iters, m, conv, rr, bb);
      if (a.trace) a.trace[(size_t)tier * a.listStride + wi] = make_uint4(m, iters, 0u, 0u);
    }
    __syncwarp();   // sInv / sLaneOf of this warp are rewritten for its next island
  }
}

// ---- dense list (kDenseSlot): islands of at most kDenseMax nodes ---------------------------------------------------------
// Once per substep: A^-1 of every island by in-place Gauss-Jordan without pivoting (A is SPD: M/h^2 sits on the diagonal).
// One 256-thread CTA per island; the matrix is assembled in shared memory from the global CSR + this substep's contact
// terms, then lives in registers (an 8 x 8 tile per thread); every elimination step broadcasts the pivot row and column
// through two small double-buffered shared arrays, one barrier per step.  fp32 is enough: the solves refine with the
// residual recomputed from the true matrix.
// N: largest island (128: 256 threads, two CTAs per SM; 192: 576 threads, one CTA per SM)
template <int N>
__global__ void __launch_bounds__((N / 8) * (N / 8), N <= 128 ? 2 : 1) k_island_invert(IslandArgs a, float* __restrict__ denseInv, int slot) {
  constexpr int kInvThreads = (N / 8) * (N / 8);
  constexpr int kInvLd = N + 4;                    // shared-memory leading dimension (floats)
  constexpr int kDenseMax = N;                     // shadows the namespace constant inside this kernel
  extern __shared__ __align__(16) unsigned char invSmem[];
  float* sA = reinterpret_cast<float*>(invSmem);
  float* sRow = sA + (size_t)kDenseMax * kInvLd;   // [2][N]
  float* sCol = sRow + 2 * kDenseMax;              // [2][N]
  const int tid = (int)threadIdx.x, ty = tid / (N / 8), tx = tid % (N / 8);
  const uint32_t count = a.counts[1 + slot];
  const uint4* descs = a.tierDesc + (size_t)slot * a.listStride;
  for (uint32_t wi = blockIdx.x; wi < count; wi += gridDim.x) {
    const uint4 desc = __ldg(descs + wi);
    const uint32_t s0 = desc.y, m = desc.z;
    const int mp = (int)((m + 7u) & ~7u);
    __syncthreads();   // the previous island's tiles are out of shared memory
    for (int i = tid; i < mp * (kInvLd / 4); i += kInvThreads) reinterpret_cast<float4*>(sA)[i] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    __syncthreads();
    if ((uint32_t)tid < m) {
      const uint32_t l = (uint32_t)tid;
      const uint32_t g = a.order[s0 + l];
      float* row = sA + (size_t)l * kInvLd;
      const uint32_t bodyBase = l - a.rankInBody[g];
      for (int kk = a.rowPtr[g]; kk < a.rowPtr[g + 1]; ++kk) {
        const uint32_t rk = __ldg(a.colRank + kk);
        if (rk != 0xffffffffu) row[bodyBase + rk] += __ldg(a.val + kk);
      }
      if (a.cPtr)
        for (int kk = a.cPtr[g]; kk < a.cPtr[g + 1]; ++kk) row[__ldg(a.pos + __ldg(a.cCol + kk)) - s0] += __ldg(a.cVal + kk);
      if (a.cDiag) row[l] += a.cDiag[g];
    }
    __syncthreads();
    const bool mine = 8 * ty < mp && 8 * tx < mp;
    float t[8][8];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const float4 lo = mine ? *reinterpret_cast<const float4*>(sA + (size_t)(8 * ty + r) * kInvLd + 8 * tx) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      const float4 hi = mine ? *reinterpret_cast<const float4*>(sA + (size_t)(8 * ty + r) * kInvLd + 8 * tx + 4) : make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      t[r][0] = lo.x; t[r][1] = lo.y; t[r][2] = lo.z; t[r][3] = lo.w; t[r][4] = hi.x; t[r][5] = hi.y; t[r][6] = hi.z; t[r][7] = hi.w;
    }
    const int nkb = mp >> 3;
    for (int kb = 0; kb < nkb; ++kb) {
#pragma unroll
      for (int kr = 0; kr < 8; ++kr) {
        const int k = 8 * kb + kr;
        if ((uint32_t)k >= m) break;   // uniform
        float* rowBuf = sRow + (k & 1) * kDenseMax;
        float* colBuf = sCol + (k & 1) * kDenseMax;
        if (ty == kb && mine) {
#pragma unroll
          for (int c = 0; c < 8; ++c) rowBuf[8 * tx + c] = t[kr][c];
        }
        if (tx == kb && mine) {
#pragma unroll
          for (int r = 0; r < 8; ++r) colBuf[8 * ty + r] = t[r][kr];
        }
        __syncthreads();
        if (mine) {
          const float d = __frcp_rn(rowBuf[k]);
          float rv[8], cv[8];
#pragma unroll
          for (int c = 0; c < 8; ++c) rv[c] = rowBuf[8 * tx + c];
#pragma unroll
          for (int r = 0; r < 8; ++r) cv[r] = colBuf[8 * ty + r] * d;
          const bool pr = ty == kb, pc = tx == kb;   // this tile holds the pivot row / column
#pragma unroll
          for (int r = 0; r < 8; ++r) {
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              float v = fmaf(-cv[r], rv[c], t[r][c]);
              if (r == kr && pr) v = rv[c] * d;
              if (c == kr && pc) v = -cv[r];
              if (r == kr && c == kr && pr && pc) v = d;
              t[r][c] = v;
            }
          }
        }
      }
    }
    if (mine) {
      float* out = denseInv + (size_t)wi * (kDenseMax * kDenseMax);
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        float4* dst = reinterpret_cast<float4*>(out + (size_t)(8 * ty + r) * kDenseMax + 8 * tx);
        dst[0] = make_float4(t[r][0], t[r][1], t[r][2], t[r][3]);
        dst[1] = make_float4(t[r][4], t[r][5], t[r][6], t[r][7]);
      }
    }
  }
}

// Every global solve: iterative refinement with the island's inverse, one 128-thread CTA per island, one row per thread.
// r = b - A x in fp64 straight from the global CSR (x gathered where it lies), then rounds of z = Ainv r (the inverse is
// symmetric: thread l reads column l, i.e. consecutive addresses across the warp; r broadcast from shared memory),
// x += z, r -= A z until the island's residual passes the tolerance.  A round contracts the residual by the accuracy of
// the fp32 inverse (1e-4 .. 1e-6), so two rounds are the rule; the round limit and the statistics are the CG tiers'.
template <int WARPS>
__device__ __forceinline__ void denseSum3(float (&v)[3], float* __restrict__ sRed, int& phase, int tid) {
#pragma unroll
  for (int k = 0; k < 3; ++k) v[k] = warpSum(v[k]);
  float* buf = sRed + phase * (4 * WARPS);
  phase ^= 1;
  if ((tid & 31) == 0) { buf[(tid >> 5) * 4 + 0] = v[0]; buf[(tid >> 5) * 4 + 1] = v[1]; buf[(tid >> 5) * 4 + 2] = v[2]; }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float t = 0.0f;
#pragma unroll
    for (int w = 0; w < WARPS; ++w) t += buf[4 * w + k];   // fixed order
    v[k] = t;
  }
}

// N: largest island = threads per CTA (128 or 192)
template <int N>
__global__ void __launch_bounds__(N, N <= 128 ? 8 : 5) k_island_dense(IslandArgs a, const float* __restrict__ denseInv, int slot) {
  constexpr int kDenseMax = N;   // shadows the namespace constant inside this kernel
  __shared__ float4 sV[N];
  __shared__ float sRed[2 * 4 * (N / 32)];
  const int tid = (int)threadIdx.x;
  const uint32_t count = a.counts[1 + slot];
  const uint4* descs = a.tierDesc + (size_t)slot * a.listStride;
  int phase = 0;
  for (uint32_t wi = blockIdx.x; wi < count; wi += gridDim.x) {
    const uint4 desc = __ldg(descs + wi);
    const uint32_t s0 = desc.y, m = desc.z;
    const long long t0 = a.trace ? clock64() : 0ll;
    const bool act = (uint32_t)tid < m;
    uint32_t g = 0, bodyBase = 0;
    int kk0 = 0, kk1 = 0, c0 = 0, c1 = 0;
    float4 xi = make_float4(0.0f, 0.0f, 0.0f, 0.0f), bi = xi;
    float cd = 0.0f;
    if (act) {
      g = a.order[s0 + tid];
      kk0 = a.rowPtr[g]; kk1 = a.rowPtr[g + 1];
      xi = a.x[g]; bi = a.b[g];
      cd = a.cDiag ? a.cDiag[g] : 0.0f;
      bodyBase = (uint32_t)tid - a.rankInBody[g];
      if (a.cPtr) { c0 = a.cPtr[g]; c1 = a.cPtr[g + 1]; }
    }
    // ---- start residual, fp64 accumulation; x of the island through shared memory (every column of an island row lies in
    //      the island: local column = body base + rank of the column, contact columns through the island permutation)
    sV[tid] = xi;
    __syncthreads();
    double y0 = (double)cd * (double)xi.x, y1 = (double)cd * (double)xi.y, y2 = (double)cd * (double)xi.z;
    for (int kk = kk0; kk < kk1; kk += 4) {   // four entries per batch: their loads are in flight together
      uint32_t rk[4]; float vv[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) if (kk + j < kk1) { rk[j] = __ldg(a.colRank + kk + j); vv[j] = __ldg(a.val + kk + j); }
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (kk + j < kk1 && rk[j] != 0xffffffffu) {
          const float4 xv = sV[bodyBase + rk[j]];
          y0 += (double)vv[j] * (double)xv.x; y1 += (double)vv[j] * (double)xv.y; y2 += (double)vv[j] * (double)xv.z;
        }
    }
    for (int kk = c0; kk < c1; ++kk) {
      const float v = a.cVal[kk];
      const float4 xv = sV[__ldg(a.pos + a.cCol[kk]) - s0];
      y0 += (double)v * (double)xv.x; y1 += (double)v * (double)xv.y; y2 += (double)v * (double)xv.z;
    }
    float r0 = 0.0f, r1 = 0.0f, r2 = 0.0f;
    if (act) { r0 = (float)((double)bi.x - y0); r1 = (float)((double)bi.y - y1); r2 = (float)((double)bi.z - y2); }
    float bb[3] = {bi.x * bi.x, bi.y * bi.y, bi.z * bi.z};
    denseSum3<N / 32>(bb, sRed, phase, tid);
    const float* inv = denseInv + (size_t)wi * (kDenseMax * kDenseMax) + tid;
    float d0 = 0.0f, d1 = 0.0f, d2 = 0.0f;
    uint32_t iters = 0;
    bool conv = false;
    float rr[3];
    while (true) {
      rr[0] = r0 * r0; rr[1] = r1 * r1; rr[2] = r2 * r2;
      denseSum3<N / 32>(rr, sRed, phase, tid);
      conv = converged3(rr, bb, a.tol2);
      if (conv || iters >= a.maxIter) break;
      sV[tid] = make_float4(r0, r1, r2, 0.0f);
      __syncthreads();
      float z0 = 0.0f, z1 = 0.0f, z2 = 0.0f;
      if (act) {
        uint32_t j = 0;
        for (; j + 8 <= m; j += 8) {
          float w[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) w[u] = __ldg(inv + (size_t)(j + u) * kDenseMax);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const float4 rj = sV[j + u];
            z0 = fmaf(w[u], rj.x, z0); z1 = fmaf(w[u], rj.y, z1); z2 = fmaf(w[u], rj.z, z2);
          }
        }
        for (; j < m; ++j) {
          const float w = __ldg(inv + (size_t)j * kDenseMax);
          const float4 rj = sV[j];
          z0 = fmaf(w, rj.x, z0); z1 = fmaf(w, rj.y, z1); z2 = fmaf(w, rj.z, z2);
        }
      }
      d0 += z0; d1 += z1; d2 += z2;
      __syncthreads();   // r has been read
      sV[tid] = make_float4(z0, z1, z2, 0.0f);
      __syncthreads();
      // r -= A z, columns through the host's rank table / the island permutation
      float w0 = cd * z0, w1 = cd * z1, w2 = cd * z2;
      for (int kk = kk0; kk < kk1; kk += 4) {
        uint32_t rk[4]; float vv[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) if (kk + j < kk1) { rk[j] = __ldg(a.colRank + kk + j); vv[j] = __ldg(a.val + kk + j); }
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (kk + j < kk1 && rk[j] != 0xffffffffu) {
            const float4 zv = sV[bodyBase + rk[j]];
            w0 = fmaf(vv[j], zv.x, w0); w1 = fmaf(vv[j], zv.y, w1); w2 = fmaf(vv[j], zv.z, w2);
          }
      }
      for (int kk = c0; kk < c1; ++kk) {
        const float v = a.cVal[kk];
        const float4 zv = sV[__ldg(a.pos + a.cCol[kk]) - s0];
        w0 = fmaf(v, zv.x, w0); w1 = fmaf(v, zv.y, w1); w2 = fmaf(v, zv.z, w2);
      }
      r0 -= w0; r1 -= w1; r2 -= w2;
      ++iters;
      // the next round's reduction barrier separates these reads of sV from its next write
    }
    if (act) {
      xi.x += d0; xi.y += d1; xi.z += d2;
      a.x[g] = xi;
    }
    if (tid == 0) {
      recordSolve(a.stats, iters, m, conv, rr, bb);
      if (a.trace) a.trace[(size_t)slot * a.listStride + wi] = make_uint4(m, iters, (uint32_t)(clock64() - t0), a.nnzOff[s0 + m] - desc.w);
    }
    __syncthreads();   // sV / sRed are reused by the CTA's next island
  }
}

// Tier 3: islands of up to a few thousand nodes (a tetrahedralised body of config 5; several toppled columns of the S3
// stack).  One 1024-thread CTA per island; r and p (what other rows gather) live in shared memory, per-row state that only
// its own thread touches (delta, A p, z) in global scratch in island order, the matrix in an island-local copy in global
// memory that stays in L2 while the CTA re-reads it every iteration, block inverses straight from the preconditioner tables.
constexpr int kBigTeam = 1024;
__global__ void __launch_bounds__(kBigTeam) k_island_pcg_big(IslandArgs a, uint32_t maxNodes, int tier) {
  extern __shared__ __align__(16) unsigned char islSmem[];
  float4* sR = reinterpret_cast<float4*>(islSmem);
  float4* sP = sR + maxNodes;
  float* sRed = reinterpret_cast<float*>(sP + maxNodes);
  const int tid = (int)threadIdx.x;
  const uint32_t count = a.counts[1 + tier];
  const uint32_t* list = a.tierList + (size_t)tier * a.listStride;
  int phase = 0;
  for (uint32_t wi = blockIdx.x; wi < count; wi += gridDim.x) {
    const uint32_t isl = list[wi];
    const uint32_t s0 = a.islStart[isl], m = a.islStart[isl + 1] - s0;
    const uint32_t z0 = a.nnzOff[s0];
    float* mv = a.matVal + z0;
    int* mc = a.matCol + z0;
    float red9[9] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
    for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
      const uint32_t g = a.order[s0 + l];
      const float4 xi = a.x[g], bi = a.b[g];
      const float cd = a.cDiag ? a.cDiag[g] : 0.0f;
      double y0 = 0.0, y1 = 0.0, y2 = 0.0;
      uint32_t e = a.nnzOff[s0 + l] - z0;
      for (int kk = a.rowPtr[g]; kk < a.rowPtr[g + 1]; ++kk, ++e) {
        const int c = __ldg(a.col + kk);
        float v = __ldg(a.val + kk);
        const float4 xv = a.x[c];
        y0 += (double)v * (double)xv.x; y1 += (double)v * (double)xv.y; y2 += (double)v * (double)xv.z;
        uint32_t lc = a.pos[c] - s0;
        if (lc >= m) { lc = l; v = 0.0f; }
        if ((uint32_t)c == g) v += cd;
        mc[e] = (int)lc; mv[e] = v;
      }
      if (a.cPtr) {
        for (int kk = a.cPtr[g]; kk < a.cPtr[g + 1]; ++kk, ++e) {
          const int c = a.cCol[kk];
          const float v = a.cVal[kk];
          const float4 xv = a.x[c];
          y0 += (double)v * (double)xv.x; y1 += (double)v * (double)xv.y; y2 += (double)v * (double)xv.z;
          mc[e] = (int)(a.pos[c] - s0); mv[e] = v;
        }
      }
      y0 += (double)cd * (double)xi.x; y1 += (double)cd * (double)xi.y; y2 += (double)cd * (double)xi.z;
      sR[l] = make_float4((float)((double)bi.x - y0), (float)((double)bi.y - y1), (float)((double)bi.z - y2), 0.0f);
      red9[6] += bi.x * bi.x; red9[7] += bi.y * bi.y; red9[8] += bi.z * bi.z;
      a.deltaScratch[s0 + l] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
      const uint32_t sl = a.slotOf[g];
      a.slotIsl[s0 + l] = sl;
      a.blkLocal[sl] = l;
    }
    __syncthreads();
    auto precond = [&](uint32_t l, float (&z)[3]) {
      const uint32_t sl = a.slotIsl[s0 + l];
      const uint32_t b = sl >> 5;
      const int lane = (int)(sl & 31u);
      const uint2 meta = a.blockMeta[b];
      const float* inv = a.blockInv + meta.x;
      const uint32_t* loc = a.blkLocal + (size_t)b * 32;
      int off = lane * (lane + 1) / 2;
      z[0] = z[1] = z[2] = 0.0f;
#pragma unroll 4
      for (int j = 0; j < (int)meta.y; ++j) {
        const float w = __ldg(inv + off);
        const float4 rj = sR[loc[j]];
        z[0] = fmaf(w, rj.x, z[0]); z[1] = fmaf(w, rj.y, z[1]); z[2] = fmaf(w, rj.z, z[2]);
        off += j < lane ? 1 : j + 1;
      }
    };
    for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
      float z[3];
      precond(l, z);
      const float4 r = sR[l];
      red9[0] += r.x * z[0]; red9[1] += r.y * z[1]; red9[2] += r.z * z[2];
      red9[3] += r.x * r.x; red9[4] += r.y * r.y; red9[5] += r.z * r.z;
      sP[l] = make_float4(z[0], z[1], z[2], 0.0f);
    }
    teamReduce<kBigTeam, 9>(red9, sRed, phase, tid);
    float rz[3] = {red9[0], red9[1], red9[2]};
    float rr[3] = {red9[3], red9[4], red9[5]};
    const float bb[3] = {red9[6], red9[7], red9[8]};
    __syncthreads();
    uint32_t iters = 0;
    bool conv = converged3(rr, bb, a.tol2);
    while (!conv && iters < a.maxIter) {
      float pap[3] = {0.0f, 0.0f, 0.0f};
      for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
        const uint32_t e0 = a.nnzOff[s0 + l] - z0, e1 = a.nnzOff[s0 + l + 1] - z0;
        float ap0 = 0.0f, ap1 = 0.0f, ap2 = 0.0f;
#pragma unroll 4
        for (uint32_t e = e0; e < e1; ++e) {
          const float v = mv[e];
          const float4 pv = sP[mc[e]];
          ap0 = fmaf(v, pv.x, ap0); ap1 = fmaf(v, pv.y, ap1); ap2 = fmaf(v, pv.z, ap2);
        }
        const float4 pl = sP[l];
        pap[0] += pl.x * ap0; pap[1] += pl.y * ap1; pap[2] += pl.z * ap2;
        a.apScratch[s0 + l] = make_float4(ap0, ap1, ap2, 0.0f);
      }
      teamReduce<kBigTeam, 3>(pap, sRed, phase, tid);
      float alpha[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) alpha[c] = pap[c] > 0.0f ? rz[c] / pap[c] : 0.0f;
      for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
        const float4 pl = sP[l], ap = a.apScratch[s0 + l], r = sR[l];
        float4 d = a.deltaScratch[s0 + l];
        d.x = fmaf(alpha[0], pl.x, d.x); d.y = fmaf(alpha[1], pl.y, d.y); d.z = fmaf(alpha[2], pl.z, d.z);
        a.deltaScratch[s0 + l] = d;
        sR[l] = make_float4(fmaf(-alpha[0], ap.x, r.x), fmaf(-alpha[1], ap.y, r.y), fmaf(-alpha[2], ap.z, r.z), 0.0f);
      }
      __syncthreads();
      float red6[6] = {0.0f, 0.0f, 0.0f, 0.0f, 0.0f, 0.0f};
      for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
        float z[3];
        precond(l, z);
        const float4 r = sR[l];
        red6[0] += r.x * z[0]; red6[1] += r.y * z[1]; red6[2] += r.z * z[2];
        red6[3] += r.x * r.x; red6[4] += r.y * r.y; red6[5] += r.z * r.z;
        a.zScratch[s0 + l] = make_float4(z[0], z[1], z[2], 0.0f);
      }
      teamReduce<kBigTeam, 6>(red6, sRed, phase, tid);
      float beta[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) { beta[c] = rz[c] > 0.0f ? red6[c] / rz[c] : 0.0f; rz[c] = red6[c]; rr[c] = red6[3 + c]; }
      ++iters;
      conv = converged3(rr, bb, a.tol2);
      if (conv) break;
      for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
        const float4 pl = sP[l], z = a.zScratch[s0 + l];
        sP[l] = make_float4(fmaf(beta[0], pl.x, z.x), fmaf(beta[1], pl.y, z.y), fmaf(beta[2], pl.z, z.z), 0.0f);
      }
      __syncthreads();
    }
    for (uint32_t l = (uint32_t)tid; l < m; l += kBigTeam) {
      const uint32_t g = a.order[s0 + l];
      float4 xv = a.x[g];
      const float4 d = a.deltaScratch[s0 + l];
      xv.x += d.x; xv.y += d.y; xv.z += d.z;
      a.x[g] = xv;
    }
    if (tid == 0) recordSolve(a.stats, iters, m, conv, rr, bb);
    __syncthreads();
  }
}

// ------------------------------------------------------------------------------------------------- host -----
namespace {
// grid of list l for `units` CTAs of work
int listGrid(int l, uint32_t units) { return (int)std::min<uint32_t>(units, (uint32_t)kLists[l].ctasPerSm * kNumSMs); }
// Test hook: PIES_B200_ISLAND_MAXBLOCKS=k shrinks the shared-memory block tables of the CG lists to k entries, so islands
// with more preconditioner blocks exercise the from-global-memory path of the block-Jacobi apply.
IslandCaps pcgCaps(int l) {
  IslandCaps c = kLists[l].caps;
  static const int forced = [] { const char* e = std::getenv("PIES_B200_ISLAND_MAXBLOCKS"); return e ? std::atoi(e) : -1; }();
  if (forced > 0 && c.maxBlocks) c.maxBlocks = std::min<uint32_t>(c.maxBlocks, (uint32_t)forced);
  return c;
}
// the arrays of the matrix, the contacts and the island order, as every island kernel reads them
IslandArgs islandArgs(const IslandWork& w, const CsrMatrix& S, const ContactLists& c) {
  IslandArgs a{};
  a.counts = w.counts.p; a.tierList = w.tierList.p; a.tierDesc = w.tierDesc.p; a.listStride = w.nBodies;
  a.islStart = w.islStart.p; a.order = w.order.p; a.pos = w.pos.p; a.nnzOff = w.nnzOff.p;
  a.rowPtr = S.rowPtr; a.col = S.col; a.val = S.val; a.colRank = w.colRank.p; a.rankInBody = w.rankInBody.p;
  a.cPtr = c.nUnique ? c.cPtr : nullptr; a.cCol = c.cCol; a.cVal = c.cVal; a.cDiag = (c.nTri || c.nodeWeights()) ? c.cDiag : nullptr;
  return a;
}
}  // namespace

#define ICHECK(expr)                                        \
  do {                                                      \
    cudaError_t _e = (expr);                                \
    if (_e != cudaSuccess) { w.lastError = _e; return -1; } \
  } while (0)

static int bitsForU(uint64_t span) { int b = 1; while ((1ull << b) <= span) ++b; return b; }

int uploadIslandStatics(IslandWork& w, cudaStream_t s, const HostSystem& y) {
  w.nBodies = y.nBodies;
  ICHECK(w.bodyOf.upload(y.bodyOf.data(), y.bodyOf.size(), s));
  ICHECK(w.rankInBody.upload(y.rankInBody.data(), y.rankInBody.size(), s));
  ICHECK(w.bodyPtr.upload(y.bodyPtr.data(), y.bodyPtr.size(), s));
  ICHECK(w.colRank.upload(y.colRank.data(), y.colRank.size(), s));
  if (!w.host) { ICHECK(cudaMallocHost(&w.host, 1024 * sizeof(uint32_t))); w.hostCap = 1024; }
  if (!w.ready) ICHECK(cudaEventCreateWithFlags(&w.ready, cudaEventDisableTiming));
  if (!w.fork) ICHECK(cudaEventCreateWithFlags(&w.fork, cudaEventDisableTiming));
  for (int k = 0; k < IslandWork::kAux; ++k) {
    if (!w.aux[k]) ICHECK(cudaStreamCreateWithFlags(&w.aux[k], cudaStreamNonBlocking));
    if (!w.join[k]) ICHECK(cudaEventCreateWithFlags(&w.join[k], cudaEventDisableTiming));
  }
  return 0;
}

int buildIslands(IslandWork& w, cudaStream_t s, uint32_t n, const CsrMatrix& S, const ContactLists& c,
                 const uint32_t* slotOf, const uint32_t* blockCount, uint32_t nBlocksBound, uint32_t tuning, int* launches) {
  int L = 0;
  const uint32_t nB = w.nBodies;
  for (uint32_t& k : w.listCount) k = 0;
  w.nLeftIslands = 0; w.nLeftNodes = 0; w.united = false;
  if (!n || !nB) return 0;
  ICHECK(w.parent.reserve(nB + 1)); ICHECK(w.keys.reserve(nB + 1)); ICHECK(w.tmpKeys.reserve(nB + 1));
  ICHECK(w.vals.reserve(nB + 1)); ICHECK(w.tmpVals.reserve(nB + 1)); ICHECK(w.heads.reserve(nB + 2));
  ICHECK(w.nodeOff.reserve(nB + 2)); ICHECK(w.posOfBody.reserve(nB + 1)); ICHECK(w.islStart.reserve(nB + 2));
  ICHECK(w.order.reserve(n + 1)); ICHECK(w.pos.reserve(n + 1)); ICHECK(w.nnzOff.reserve(n + 2));
  ICHECK(w.tierList.reserve((size_t)(kIslandLists + 1) * nB)); ICHECK(w.tierDesc.reserve((size_t)(kIslandLists + 1) * nB)); ICHECK(w.counts.reserve(16));
  ICHECK(w.blkLocal.reserve((size_t)nBlocksBound * 32 + 32)); ICHECK(w.slotIsl.reserve(n + 1));
  static const bool traceOn = std::getenv("PIES_B200_ISLAND_TRACE") != nullptr;
  if (traceOn) ICHECK(w.trace.reserve((size_t)(kIslandLists + 1) * nB));
  ICHECK(w.sortHist.reserve(sortHistBytes(nB) / 4 + 4));
  w.scanCap = std::max<uint64_t>(w.scanCap, std::max<uint64_t>(n, nB) + 2);
  ICHECK(w.scanScratch.reserve(scanScratchElems(w.scanCap)));
  ICHECK(cudaMemsetAsync(w.counts.p, 0, 16 * sizeof(uint32_t), s));
  const int united = c.nUnique ? 1 : 0;
  w.united = united != 0;
  if (united) {
    k_isl_init<<<gridFor(nB, kThreads), kThreads, 0, s>>>(nB, w.parent.p); ++L;
    k_isl_unite<<<gridFor(c.nUnique, kThreads), kThreads, 0, s>>>(c.nUnique, c.uTri, w.bodyOf.p, w.parent.p); ++L;
  }
  k_isl_keys<<<gridFor(nB, kThreads), kThreads, 0, s>>>(nB, w.parent.p, united, w.keys.p, w.vals.p); ++L;
  if (united) L += launchSortPairs(s, nB, w.keys.p, w.vals.p, w.tmpKeys.p, w.tmpVals.p, w.sortHist.p, bitsForU(nB));
  k_isl_heads<<<gridFor(nB + 1, kThreads), kThreads, 0, s>>>(nB, w.keys.p, w.vals.p, w.bodyPtr.p, w.heads.p, w.nodeOff.p,
                                                            w.posOfBody.p); ++L;
  L += launchExclusiveScan(s, w.heads.p, nB + 1, w.scanScratch.p);
  L += launchExclusiveScan(s, w.nodeOff.p, nB + 1, w.scanScratch.p);
  k_isl_starts<<<gridFor(nB, kThreads), kThreads, 0, s>>>(nB, n, w.keys.p, w.heads.p, w.nodeOff.p, w.islStart.p, w.counts.p); ++L;
  k_isl_nodes<<<gridFor(n + 1, kThreads), kThreads, 0, s>>>(n, w.bodyOf.p, w.rankInBody.p, w.posOfBody.p, w.nodeOff.p, S.rowPtr,
                                                           c.nUnique ? c.cPtr : nullptr, w.order.p, w.pos.p, w.nnzOff.p); ++L;
  L += launchExclusiveScan(s, w.nnzOff.p, n + 1, w.scanScratch.p);
  static const uint32_t switchedOff = (std::getenv("PIES_B200_NO_SMALL_CTA") ? kNoSmallCta : 0u) |
                                      (std::getenv("PIES_B200_NO_DENSE") ? kNoDense : 0u) |
                                      (std::getenv("PIES_B200_NO_DENSE2") ? kNoDense2 : 0u);
  IslandClassifyTable tt;
  for (int o = 0; o < kIslandLists; ++o) {
    tt.id[o] = kClassifyOrder[o];
    tt.list[o] = kLists[tt.id[o]];
    if (tt.list[o].offBy & switchedOff) tt.list[o].caps.maxNodes = 0;
  }
  // Tuning bits: 4 = no island-local solve, 16 << t = public tier t off, 256 = tier 3 on.  Tier 3 is opt-in: a handful of
  // its islands keep single SMs busy for milliseconds, the grid-wide CG spreads them over the whole device.
  const uint32_t avail = (tuning & 256u) ? 0xFu : 0x7u;
  tt.tiersOn = (tuning & 4u) ? 0u : (avail & ~((tuning >> 4) & 0xFu));
  k_isl_classify<<<gridFor(nB, kThreads), kThreads, 0, s>>>(w.counts.p, tt, w.islStart.p, w.nnzOff.p, w.order.p, slotOf, blockCount,
                                                           nB, w.tierList.p, w.tierDesc.p, w.counts.p); ++L;
  ICHECK(cudaMemcpyAsync(w.host, w.counts.p, 12 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  ICHECK(cudaEventRecord(w.ready, s));
  ICHECK(cudaEventSynchronize(w.ready));
  for (int l = 0; l < kIslandLists; ++l) w.listCount[l] = w.host[1 + l];
  w.nLeftIslands = w.host[1 + kIslandLists];
  w.nLeftNodes = w.host[2 + kIslandLists];
  w.inverseFloats = w.host[3 + kIslandLists];
  // Both kinds present: the grid-wide CG only has to run over the rows of the left-over islands.
  w.restricted = false;
  if (w.nLeftIslands && w.anyLocal()) {
    const uint32_t nWin = (n + 255u) / 256u;
    ICHECK(w.big.reserve(n + 1)); ICHECK(w.winFlag.reserve(nWin + 2)); ICHECK(w.blkFlag.reserve(nBlocksBound + 2));
    ICHECK(w.actWin.reserve(nWin + 1)); ICHECK(w.actBlk.reserve(nBlocksBound + 1)); ICHECK(w.actCounts.reserve(4));
    w.scanCap = std::max<uint64_t>(w.scanCap, std::max<uint64_t>(nWin, nBlocksBound) + 2);
    ICHECK(w.scanScratch.reserve(scanScratchElems(w.scanCap)));
    ICHECK(cudaMemsetAsync(w.big.p, 0, n + 1, s));
    ICHECK(cudaMemsetAsync(w.winFlag.p, 0, (nWin + 2) * sizeof(uint32_t), s));
    ICHECK(cudaMemsetAsync(w.blkFlag.p, 0, ((size_t)nBlocksBound + 2) * sizeof(uint32_t), s));
    k_isl_mark_big<<<(int)std::min<uint32_t>(w.nLeftIslands, 4 * kNumSMs), kThreads, 0, s>>>(
        w.counts.p, w.tierList.p + (size_t)kIslandLists * nB, w.islStart.p, w.order.p, slotOf, w.big.p, w.winFlag.p, w.blkFlag.p); ++L;
    L += launchExclusiveScan(s, w.winFlag.p, nWin + 1, w.scanScratch.p);
    k_isl_compact<<<gridFor(nWin + 1, kThreads), kThreads, 0, s>>>(nWin, w.winFlag.p, w.actWin.p, w.actCounts.p); ++L;
    L += launchExclusiveScan(s, w.blkFlag.p, (uint64_t)nBlocksBound + 1, w.scanScratch.p);
    k_isl_compact<<<gridFor((uint64_t)nBlocksBound + 1, kThreads), kThreads, 0, s>>>(nBlocksBound, w.blkFlag.p, w.actBlk.p, w.actCounts.p + 1); ++L;
    w.restricted = true;
  }
  // What the lists need before the first solve of the substep, in launch order (the longer inversions first)
  const IslandArgs a = islandArgs(w, S, c);
  for (const int l : kLaunchOrder) {
    const uint32_t count = w.listCount[l], N = kLists[l].caps.maxNodes;
    if (!count) continue;
    if (kLists[l].kind == kBig) {   // an island-local copy of the matrix in global memory
      const size_t nnz = S.nnz + 6ull * c.nUnique + 16;
      ICHECK(w.matCol.reserve(nnz)); ICHECK(w.matVal.reserve(nnz));
    } else if (kLists[l].kind == kDense) {
      // The inverses, on the solver's stream: run beside the first local step on a side stream (r02x) they only moved
      // their time from one phase to the other — both want every SM — and blurred the per-kernel timings of that step.
      // One CTA of (N/8)^2 threads per island, as many per SM as the kernel's launch bounds.
      ICHECK(w.denseInv[l].reserve((size_t)count * N * N));
      const auto kernel = N == kDenseMax ? k_island_invert<(int)kDenseMax> : k_island_invert<(int)kDenseMax2>;
      const size_t smem = ((size_t)N * (N + 4) + 4 * N) * sizeof(float);
      cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
      kernel<<<(int)std::min<uint32_t>(count, (N <= 128 ? 2 : 1) * kNumSMs), (N / 8) * (N / 8), smem, s>>>(a, w.denseInv[l].p, l); ++L;
    }
  }
  if (launches) *launches += L;
  return 0;
}

void islandStats(const IslandWork& w, PiesB200Stats& st) {
  for (uint32_t& k : st.islandsTier) k = 0;
  for (int l = 0; l < kIslandLists; ++l) st.islandsTier[kLists[l].tier] += w.listCount[l];
  st.islandsGlobal = w.nLeftIslands;
  st.islandNodesGlobal = w.nLeftNodes;
  st.islandInverseFloats = w.inverseFloats;
}

int launchIslandSolve(IslandWork& w, cudaStream_t s, const CsrMatrix& S, const ContactLists& c, const PcgWork& pw,
                      const uint32_t* slotOf, const float4* b, float4* x, float tol, uint32_t maxIter, uint32_t statSlot) {
  IslandArgs a = islandArgs(w, S, c);
  a.slotOf = slotOf; a.blockNodes = pw.blockNodes; a.blockInv = pw.blockInv; a.blockMeta = pw.blockMeta;
  a.blkLocal = w.blkLocal.p; a.matCol = w.matCol.p; a.matVal = w.matVal.p; a.deltaScratch = pw.delta;
  a.apScratch = pw.ap; a.zScratch = pw.z; a.slotIsl = w.slotIsl.p;
  a.b = b; a.x = x; a.tol2 = tol * tol; a.maxIter = maxIter; a.stats = w.solveStats.p + 4ull * statSlot;
  a.trace = w.trace.p;   // null unless PIES_B200_ISLAND_TRACE reserved it
  int L = 0;
  // The lists of one solve are independent: the first one enqueued runs on the solver's stream, every further one on a
  // stream of its own beside it (the handful of long-running islands of tiers 2 and 3 next to the thousands of small ones
  // that fill the other SMs; the warp list in the SMs a CTA list's last, partly filled wave leaves idle).
  int present = 0;
  for (uint32_t k : w.listCount) present += k ? 1 : 0;
  if (present > 1) cudaEventRecord(w.fork, s);   // before anything of this solve is enqueued on s
  int used = 0;
  for (const int l : kLaunchOrder) {
    const uint32_t count = w.listCount[l];
    if (!count) continue;
    cudaStream_t st = s;   // the first list enqueued
    if (L) { st = w.aux[used++]; cudaStreamWaitEvent(st, w.fork, 0); }
    const IslandList& e = kLists[l];
    switch (e.kind) {
      case kDirect:   // eight warps per CTA
        k_island_direct<<<listGrid(l, (count + 7) / 8), 256, 0, st>>>(a, l);
        break;
      case kDense: {
        const auto kernel = e.caps.maxNodes == kDenseMax ? k_island_dense<(int)kDenseMax> : k_island_dense<(int)kDenseMax2>;
        kernel<<<listGrid(l, count), e.team, 0, st>>>(a, w.denseInv[l].p, l);
        break;
      }
      case kCtaCg: {   // t: the list whose team, shared-memory layout and caps solve list l
        const int t = count <= (uint32_t)kLists[e.shortList].ctasPerSm * kNumSMs ? e.shortList : l;
        const IslandList& h = kLists[t];
        const auto kernel = h.team == 128 ? k_island_pcg<128, 2> : (h.team == 320 ? k_island_pcg<320, 2> : k_island_pcg<512, 2>);
        const IslandLayout lay = islandLayout(h.caps);
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lay.total);
        kernel<<<listGrid(t, count), h.team, lay.total, st>>>(a, lay, pcgCaps(t), l);
        break;
      }
      case kBig: {
        const size_t smem = 32ull * e.caps.maxNodes + 2 * 9 * 32 * sizeof(float);
        cudaFuncSetAttribute(k_island_pcg_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        k_island_pcg_big<<<listGrid(l, count), kBigTeam, smem, st>>>(a, e.caps.maxNodes, l);
        break;
      }
    }
    ++L;
  }
  for (int k = 0; k < used; ++k) { cudaEventRecord(w.join[k], w.aux[k]); cudaStreamWaitEvent(s, w.join[k], 0); }
  return L;
}

void applyRestriction(const IslandWork& w, PcgWork& pw) {
  if (!w.restricted) return;
  pw.big = w.big.p; pw.actWin = w.actWin.p; pw.actBlk = w.actBlk.p; pw.actCounts = w.actCounts.p;
}

void preloadIslandKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_isl_mark_big);
  cudaFuncGetAttributes(&a, k_isl_compact);
  cudaFuncGetAttributes(&a, k_isl_init);
  cudaFuncGetAttributes(&a, k_isl_unite);
  cudaFuncGetAttributes(&a, k_isl_keys);
  cudaFuncGetAttributes(&a, k_isl_heads);
  cudaFuncGetAttributes(&a, k_isl_starts);
  cudaFuncGetAttributes(&a, k_isl_nodes);
  cudaFuncGetAttributes(&a, k_isl_classify);
  cudaFuncGetAttributes(&a, k_island_pcg<320, 2>);
  cudaFuncGetAttributes(&a, k_island_pcg<128, 2>);
  cudaFuncGetAttributes(&a, k_island_pcg<512, 2>);
  cudaFuncGetAttributes(&a, k_island_pcg_big);
  cudaFuncGetAttributes(&a, k_island_direct);
  cudaFuncGetAttributes(&a, k_island_invert<(int)kDenseMax>);
  cudaFuncGetAttributes(&a, k_island_invert<(int)kDenseMax2>);
  cudaFuncGetAttributes(&a, k_island_dense<(int)kDenseMax>);
  cudaFuncGetAttributes(&a, k_island_dense<(int)kDenseMax2>);
}

}  // namespace pies
