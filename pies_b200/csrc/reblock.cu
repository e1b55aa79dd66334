// reblock.cu — contact-aware block-Jacobi preconditioner, rebuilt once per substep.
//
// The reference re-factorises S + C_t every substep (reference Src/Solver.cpp:242-262); the CG that
// replaces it only needs a preconditioner, but it must see the collision terms: a point-triangle
// constraint carries copies * 1e4 against ~1e4 of elastic stiffness, so four nodes joined by a contact
// move almost rigidly together and a per-body block (which cuts the contact) leaves a condition number
// of ~100 (60-80 CG iterations).  Here the nodes joined by contacts are taken out of their static block
// and regrouped into "contact clusters" (connected components of the contact graph, cut into spatially
// compact pieces of <= 32 nodes), so every contact lies inside one dense block; what is left of the
// static blocks is re-inverted without the removed nodes.  Measured on the reference's own matrices
// (tick 61 / tick 110 of the S3 stack): 68 -> 18 and 82 -> 32 iterations at 1e-7.
//
// Pipeline (all on the solver stream, one host read of the touched-node count):
//   touched flags -> ordered compaction -> union-find roots -> sort by (root, Morton code) ->
//   cluster starts -> block offsets -> membership tables -> per-warp dense Cholesky inverse.
#include "reblock.h"

#include "common.cuh"

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- touched nodes -----------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_touched_flags(uint32_t n, const int* __restrict__ incPtr,
                                                            uint32_t* __restrict__ flag, uint32_t* __restrict__ parent) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  if (i == n) { flag[i] = 0; return; }
  flag[i] = incPtr[i + 1] > incPtr[i] ? 1u : 0u;
  parent[i] = i;
}

// ---- min-id union-find over the contact graph -------------------------------------------------------
__device__ __forceinline__ uint32_t ufFind(uint32_t* parent, uint32_t x) {
  uint32_t p = *(volatile uint32_t*)(parent + x);
  while (p != x) { x = p; p = *(volatile uint32_t*)(parent + x); }
  return x;
}

__device__ __forceinline__ void ufUnite(uint32_t* parent, uint32_t u, uint32_t v) {
  while (true) {
    u = ufFind(parent, u);
    v = ufFind(parent, v);
    if (u == v) return;
    if (u < v) { uint32_t t = u; u = v; v = t; }  // hook the larger root under the smaller one
    uint32_t old = atomicMin(parent + u, v);
    if (old == u) return;
    u = old;  // someone re-parented u meanwhile: merge what it points to with v
  }
}

__global__ void __launch_bounds__(kThreads) k_uf_unite(uint32_t nU, const uint4* __restrict__ entries,
                                                       uint32_t* __restrict__ parent) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nU) return;
  uint4 id = entries[e];
  ufUnite(parent, id.x, id.y);
  ufUnite(parent, id.x, id.z);
  ufUnite(parent, id.x, id.w);
}

// (root, Morton code of the position) keys of the touched nodes, emitted in ascending node order
__device__ __forceinline__ uint32_t spread5(uint32_t v) {  // 5 bits -> every third bit
  v &= 31u;
  v = (v | (v << 8)) & 0x100Fu;
  v = (v | (v << 4)) & 0x10C3u;
  v = (v | (v << 2)) & 0x1249u;
  return v;
}

__global__ void __launch_bounds__(kThreads) k_touched_keys(uint32_t n, const uint32_t* __restrict__ flagScan,
                                                           uint32_t* __restrict__ parent, const float4* __restrict__ q,
                                                           uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint32_t pos = flagScan[i];
  if (flagScan[i + 1] == pos) return;  // not touched
  uint32_t root = ufFind(parent, i);
  float4 p = q[i];
  // half-unit cells, wrapping every 16 units: only used to keep the pieces of a large cluster compact
  uint32_t mx = (uint32_t)(int)floorf(p.x * 2.0f), my = (uint32_t)(int)floorf(p.y * 2.0f), mz = (uint32_t)(int)floorf(p.z * 2.0f);
  uint32_t morton = spread5(mx) | (spread5(my) << 1) | (spread5(mz) << 2);
  keys[pos] = ((uint64_t)root << 15) | morton;
  vals[pos] = i;
}

__global__ void __launch_bounds__(kThreads) k_cluster_heads(uint32_t nT, const uint64_t* __restrict__ keys,
                                                            uint32_t* __restrict__ heads) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j > nT) return;
  heads[j] = (j < nT && (j == 0 || (keys[j] >> 15) != (keys[j - 1] >> 15))) ? 1u : 0u;
}

// cluster index per sorted position (in place of the scanned heads) and cluster starts
__global__ void __launch_bounds__(kThreads) k_cluster_starts(uint32_t nT, const uint64_t* __restrict__ keys,
                                                             uint32_t* __restrict__ headScan, uint32_t* __restrict__ start) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nT) return;
  bool head = (j == 0 || (keys[j] >> 15) != (keys[j - 1] >> 15));
  uint32_t idx = headScan[j] + (head ? 1u : 0u) - 1u;
  if (head) start[idx] = j;
  if (j == nT - 1) start[idx + 1] = nT;
  headScan[j] = idx;
}

// blocks per cluster (to be scanned); entry [nClusters] = 0
__global__ void __launch_bounds__(kThreads) k_cluster_blocks(uint32_t nT, const uint32_t* __restrict__ nClustersPtr,
                                                             const uint32_t* __restrict__ start, uint32_t* __restrict__ nb) {
  uint32_t c = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t nC = *nClustersPtr;
  if (c > nC || c > nT) return;
  nb[c] = c < nC ? (start[c + 1] - start[c] + 31u) / 32u : 0u;
}

__global__ void __launch_bounds__(kThreads) k_assign_dynamic(uint32_t nT, uint32_t nStatic,
                                                             const uint32_t* __restrict__ nClustersPtr,
                                                             const uint32_t* __restrict__ clusterIdx,
                                                             const uint32_t* __restrict__ start,
                                                             const uint32_t* __restrict__ blkOff,
                                                             const uint32_t* __restrict__ nodes, int* __restrict__ blockNodes,
                                                             uint32_t* __restrict__ slotOf, uint32_t* __restrict__ blockCount,
                                                             uint32_t* __restrict__ clusterOf, uint8_t* __restrict__ gsClass,
                                                             uint32_t* __restrict__ rankOf, uint32_t* __restrict__ midList,
                                                             uint32_t* __restrict__ midCount, uint32_t midMax,
                                                             uint32_t* __restrict__ nBlocksOut) {
  uint32_t j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j == 0) *nBlocksOut = nStatic + (nT ? blkOff[*nClustersPtr] : 0u);
  if (j >= nT) return;
  uint32_t c = clusterIdx[j];
  uint32_t rank = j - start[c];
  uint32_t blk = nStatic + blkOff[c] + (rank >> 5);
  uint32_t slot = blk * 32u + (rank & 31u);
  blockNodes[slot] = (int)nodes[j];
  slotOf[nodes[j]] = slot;
  const uint32_t size = start[c + 1] - start[c];
  clusterOf[nodes[j]] = c;
  rankOf[nodes[j]] = rank;
  // 1: the whole cluster is one block (in-warp ordered sweeps from registers), 3: one warp sweeps it from shared
  // memory, 2: dataflow sweeps
  gsClass[nodes[j]] = size <= 32u ? 1 : (size <= midMax ? 3 : 2);
  if (rank == 0u && size > 32u) {
    if (size <= midMax) midList[atomicAdd(midCount, 1u)] = c;  // order irrelevant: clusters are independent
    else atomicAdd(midCount + 1, 1u);
  }
  if ((rank & 31u) == 0u) blockCount[blk] = min(32u, size - rank);
}

// storage of every block's inverse: the lower triangle of the symmetric m x m matrix, packed by rows
// (m (m + 1) / 2 floats, rounded up to 16 B; entry (j, i), i <= j, at j (j + 1) / 2 + i), offsets by exclusive scan
__global__ void __launch_bounds__(kThreads) k_block_sizes(uint32_t bound, const uint32_t* __restrict__ nBlocksPtr,
                                                          const uint32_t* __restrict__ blockCount, uint32_t* __restrict__ sq) {
  uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b > bound) return;
  uint32_t m = b < *nBlocksPtr ? blockCount[b] : 0u;
  sq[b] = (m * (m + 1u) / 2u + 3u) & ~3u;
}

// static blocks: drop the touched nodes and pack the rest to the front (one warp per block)
__global__ void __launch_bounds__(kThreads) k_static_membership(uint32_t nStatic, const int* __restrict__ staticNodes,
                                                                const uint32_t* __restrict__ flagScan,
                                                                const float* __restrict__ floorW, int haveFloor,
                                                                int* __restrict__ blockNodes, uint32_t* __restrict__ slotOf,
                                                                uint32_t* __restrict__ blockCount, uint8_t* __restrict__ dirty) {
  uint32_t b = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  int lane = threadIdx.x & 31;
  if (b >= nStatic) return;
  int node = staticNodes[b * 32 + lane];
  bool present = node >= 0;
  bool keep = present && flagScan[node + 1] == flagScan[node];
  bool floorNode = keep && haveFloor && floorW[node] != 0.0f;
  uint32_t keepMask = __ballot_sync(0xffffffffu, keep);
  uint32_t presentMask = __ballot_sync(0xffffffffu, present);
  uint32_t floorMask = __ballot_sync(0xffffffffu, floorNode);
  blockNodes[b * 32 + lane] = -1;
  __syncwarp();
  if (keep) {
    uint32_t dst = b * 32 + __popc(keepMask & ((1u << lane) - 1u));
    blockNodes[dst] = node;
    slotOf[node] = dst;
  }
  if (lane == 0) {
    dirty[b] = (keepMask != presentMask || floorMask != 0u) ? 1 : 0;
    blockCount[b] = __popc(keepMask);
  }
}

// ---- dense assembly + Cholesky inverse, one warp per block ----------------------------------------------
constexpr int kFactorWarps = 4;
constexpr int kLd = 33;

__global__ void __launch_bounds__(kFactorWarps * 32) k_block_factor(uint32_t nStatic, const uint32_t* __restrict__ nBlocksPtr,
                                                                    CsrMatrix S, ContactLists c,
                                                                    const int* __restrict__ blockNodes,
                                                                    const uint32_t* __restrict__ slotOf,
                                                                    const uint8_t* __restrict__ dirty,
                                                                    const uint32_t* __restrict__ blockOff,
                                                                    const float* __restrict__ baseInv,
                                                                    float* __restrict__ blockInv, uint2* __restrict__ blockMeta) {
  __shared__ float sM[kFactorWarps][32 * kLd];
  __shared__ float sX[kFactorWarps][32 * kLd];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t b = blockIdx.x * kFactorWarps + warp;
  if (b >= *nBlocksPtr) return;
  float* out = blockInv + blockOff[b];
  const int node = blockNodes[b * 32 + lane];
  const uint32_t valid = __ballot_sync(0xffffffffu, node >= 0);
  const int m = __popc(valid);  // members are packed at the front; the inverse is stored as a packed lower triangle
  if (lane == 0) blockMeta[b] = make_uint2(blockOff[b], (uint32_t)m);
  if (b < nStatic && !dirty[b]) {  // untouched static block: the once-per-topology inverse (stored 32 x 32)
    const float* src = baseInv + (size_t)b * 1024;
    for (int j = 0; j < m; ++j) if (lane <= j) out[j * (j + 1) / 2 + lane] = src[j * 32 + lane];
    return;
  }
  float* M = sM[warp];
  float* X = sX[warp];
  for (int k = 0; k < 32; ++k) { M[k * kLd + lane] = 0.0f; X[k * kLd + lane] = 0.0f; }
  __syncwarp();
  if (node >= 0) {
    float* row = M + lane * kLd;
    for (int k = S.rowPtr[node]; k < S.rowPtr[node + 1]; ++k) {
      uint32_t sj = slotOf[S.col[k]];
      if ((sj >> 5) == b) row[sj & 31u] = S.val[k];
    }
    float diag = row[lane];
    if (c.nodeWeights()) diag += c.floorW[node];
    if (c.nUnique) {
      for (int k = c.incPtr[node]; k < c.incPtr[node + 1]; ++k) {
        uint32_t v = c.inc[k];
        uint4 e = c.uTri[v >> 2];
        float wgt = c.uW[v >> 2];
        if ((v & 3u) == 0u) {
          diag += 3.0f * wgt;
          uint32_t sb = slotOf[e.y], sc = slotOf[e.z], sd = slotOf[e.w];
          if ((sb >> 5) == b) row[sb & 31u] -= wgt;
          if ((sc >> 5) == b) row[sc & 31u] -= wgt;
          if ((sd >> 5) == b) row[sd & 31u] -= wgt;
        } else {
          diag += wgt;
          uint32_t sa = slotOf[e.x];
          if ((sa >> 5) == b) row[sa & 31u] -= wgt;
        }
      }
    }
    row[lane] = diag;
  }
  __syncwarp();
  // Cholesky, left-looking by columns: lane i owns row i
  bool ok = true;
  for (int j = 0; j < m; ++j) {
    float s = 0.0f;
    if (lane >= j && lane < m) {
      s = M[lane * kLd + j];
      for (int k = 0; k < j; ++k) s -= M[lane * kLd + k] * M[j * kLd + k];
    }
    float d = __shfl_sync(0xffffffffu, s, j);
    if (!(d > 0.0f)) { ok = false; break; }
    d = sqrtf(d);
    if (lane >= j && lane < m) M[lane * kLd + j] = lane == j ? d : s / d;
    __syncwarp();
  }
  if (!ok) {  // not SPD in fp32 (should not happen: M/h^2 sits on the diagonal): Jacobi for this block
    __syncwarp();
    float diag = 1.0f;
    if (node >= 0) {
      for (int k = S.rowPtr[node]; k < S.rowPtr[node + 1]; ++k) if (S.col[k] == node) diag = S.val[k];
    }
    for (int j = 0; j < m; ++j) if (lane <= j) out[j * (j + 1) / 2 + lane] = j == lane ? 1.0f / diag : 0.0f;
    return;
  }
  // X = L^-1 (lower): lane c owns column c
  if (lane < m) {
    X[lane * kLd + lane] = 1.0f / M[lane * kLd + lane];
    for (int i = lane + 1; i < m; ++i) {
      float s = 0.0f;
      for (int k = lane; k < i; ++k) s -= M[i * kLd + k] * X[k * kLd + lane];
      X[i * kLd + lane] = s / M[i * kLd + i];
    }
  }
  __syncwarp();
  // Minv = X^T X, lower triangle only: lane i <= j owns entry (j, i)
  for (int j = 0; j < m; ++j) {
    if (lane <= j) {
      float s = 0.0f;
      for (int k = j; k < m; ++k) s += X[k * kLd + lane] * X[k * kLd + j];
      out[j * (j + 1) / 2 + lane] = s;
    }
  }
}

#define RCHECK(expr)                                       \
  do {                                                     \
    cudaError_t _e = (expr);                               \
    if (_e != cudaSuccess) { w.lastError = _e; return -1; } \
  } while (0)

static int bitsForU(uint64_t span) { int b = 1; while ((1ull << b) <= span) ++b; return b; }

int rebuildBlocks(BlockWork& w, cudaStream_t s, uint32_t n, const CsrMatrix& S, const int* staticNodes,
                  const float* staticInv, uint32_t nStatic, const ContactLists& c, const float4* q, PcgWork& pw,
                  int* launches) {
  int L = 0;
  if (w.factorPending) { RCHECK(cudaStreamWaitEvent(s, w.factorDone, 0)); w.factorPending = false; }  // an aborted substep's inversions
  RCHECK(w.nBlocksDev.reserve(4));
  RCHECK(w.flag.reserve(n + 2)); RCHECK(w.parent.reserve(n + 1)); RCHECK(w.slotOf.reserve(n + 1));
  RCHECK(w.dirty.reserve(nStatic + 1));
  RCHECK(w.clusterOf.reserve(n + 1)); RCHECK(w.gsClass.reserve(n + 1)); RCHECK(w.rankOf.reserve(n + 1));
  RCHECK(w.midCount.reserve(4));
  RCHECK(cudaMemsetAsync(w.midCount.p, 0, 4 * sizeof(uint32_t), s));
  if (!w.countsReady) RCHECK(cudaEventCreateWithFlags(&w.countsReady, cudaEventDisableTiming));
  RCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(n + 2, w.scanCap))));
  RCHECK(cudaMemsetAsync(w.gsClass.p, 0, n + 1, s));
  uint32_t nT = 0;
  if (c.nUnique) {
    k_touched_flags<<<gridFor(n + 1, kThreads), kThreads, 0, s>>>(n, c.incPtr, w.flag.p, w.parent.p); ++L;
    L += launchExclusiveScan(s, w.flag.p, n + 1, w.scanScratch.p);
    RCHECK(cudaMemcpyAsync(w.host, w.flag.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    k_uf_unite<<<gridFor(c.nUnique, kThreads), kThreads, 0, s>>>(c.nUnique, c.uTri, w.parent.p); ++L;
    RCHECK(cudaStreamSynchronize(s));
    nT = w.host[0];
  } else {
    RCHECK(cudaMemsetAsync(w.flag.p, 0, (n + 2) * sizeof(uint32_t), s));
  }
  // every cluster has >= 4 nodes (a contact joins 4 distinct nodes): #clusters <= nT / 4, #pieces <= that + nT / 32
  uint32_t dynBound = nT ? nT / 4 + nT / 32 + 2 : 0;
  uint32_t bound = nStatic + dynBound;
  w.nBlocksBound = bound;
  RCHECK(w.blockNodes.reserve((size_t)bound * 32));
  RCHECK(w.blockCount.reserve(bound + 2)); RCHECK(w.blockOff.reserve(bound + 2)); RCHECK(w.blockMeta.reserve(bound + 2));
  RCHECK(w.blockInv.reserve((size_t)17 * n + 4ull * bound + 64));  // sum m (m + 1) / 2 <= 16.5 * sum m, plus rounding
  w.scanCap = std::max<uint64_t>(w.scanCap, (uint64_t)bound + 2);
  if (nT) {
    RCHECK(w.keys.reserve(nT)); RCHECK(w.tmpKeys.reserve(nT)); RCHECK(w.vals.reserve(nT)); RCHECK(w.tmpVals.reserve(nT));
    RCHECK(w.heads.reserve(nT + 2)); RCHECK(w.start.reserve(nT + 2)); RCHECK(w.blkOff.reserve(nT + 2));
    RCHECK(w.midList.reserve(nT / 33 + 2));
    RCHECK(w.sortHist.reserve(sortHistBytes(nT) / 4 + 4));
    w.scanCap = std::max<uint64_t>(w.scanCap, (uint64_t)nT + 2);
    RCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(n + 2, w.scanCap))));
    RCHECK(cudaMemsetAsync(w.blockNodes.p + (size_t)nStatic * 32, 0xff, (size_t)dynBound * 32 * sizeof(int), s));
    RCHECK(cudaMemsetAsync(w.blockCount.p + nStatic, 0, (size_t)(dynBound + 1) * sizeof(uint32_t), s));
    k_touched_keys<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, w.flag.p, w.parent.p, q, w.keys.p, w.vals.p); ++L;
    L += launchSortPairs(s, nT, w.keys.p, w.vals.p, w.tmpKeys.p, w.tmpVals.p, w.sortHist.p, bitsForU(n) + 15);
    k_cluster_heads<<<gridFor(nT + 1, kThreads), kThreads, 0, s>>>(nT, w.keys.p, w.heads.p); ++L;
    L += launchExclusiveScan(s, w.heads.p, nT + 1, w.scanScratch.p);
    k_cluster_starts<<<gridFor(nT, kThreads), kThreads, 0, s>>>(nT, w.keys.p, w.heads.p, w.start.p); ++L;
    k_cluster_blocks<<<gridFor(nT + 1, kThreads), kThreads, 0, s>>>(nT, w.heads.p + nT, w.start.p, w.blkOff.p); ++L;
    L += launchExclusiveScan(s, w.blkOff.p, nT + 1, w.scanScratch.p);  // entries past #clusters are unused
  } else {
    RCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(n + 2, w.scanCap))));
  }
  k_static_membership<<<gridFor((uint64_t)nStatic * 32, kThreads), kThreads, 0, s>>>(nStatic, staticNodes, w.flag.p, c.floorW,
                                                                                    c.nodeWeights() ? 1 : 0, w.blockNodes.p,
                                                                                    w.slotOf.p, w.blockCount.p, w.dirty.p); ++L;
  k_assign_dynamic<<<gridFor(std::max(nT, 1u), kThreads), kThreads, 0, s>>>(nT, nStatic, w.heads.p + nT, w.heads.p, w.start.p,
                                                                           w.blkOff.p, w.vals.p, w.blockNodes.p, w.slotOf.p,
                                                                           w.blockCount.p, w.clusterOf.p, w.gsClass.p,
                                                                           w.rankOf.p, w.midList.p, w.midCount.p, w.midClusterMax,
                                                                           w.nBlocksDev.p); ++L;
  RCHECK(cudaMemcpyAsync(w.host + 1, w.midCount.p, 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  RCHECK(cudaEventRecord(w.countsReady, s));
  k_block_sizes<<<gridFor(bound + 1, kThreads), kThreads, 0, s>>>(bound, w.nBlocksDev.p, w.blockCount.p, w.blockOff.p); ++L;
  L += launchExclusiveScan(s, w.blockOff.p, bound + 1, w.scanScratch.p);
  if (!w.side) {
    RCHECK(cudaStreamCreateWithFlags(&w.side, cudaStreamNonBlocking));
    RCHECK(cudaEventCreateWithFlags(&w.factorFork, cudaEventDisableTiming));
    RCHECK(cudaEventCreateWithFlags(&w.factorDone, cudaEventDisableTiming));
  }
  RCHECK(cudaEventRecord(w.factorFork, s));
  RCHECK(cudaStreamWaitEvent(w.side, w.factorFork, 0));
  k_block_factor<<<gridFor(bound, kFactorWarps), kFactorWarps * 32, 0, w.side>>>(nStatic, w.nBlocksDev.p, S, c, w.blockNodes.p,
                                                                                w.slotOf.p, w.dirty.p, w.blockOff.p, staticInv,
                                                                                w.blockInv.p, w.blockMeta.p); ++L;
  RCHECK(cudaEventRecord(w.factorDone, w.side));
  w.factorPending = true;
  pw.blockNodes = w.blockNodes.p; pw.blockInv = w.blockInv.p; pw.blockMeta = w.blockMeta.p; pw.nBlocks = bound;
  pw.nBlocksDev = w.nBlocksDev.p;
  w.nTouched = nT;
  if (launches) *launches += L;
  return 0;
}

// Loads this file's kernels now (CUDA loads a kernel lazily at its first launch; for the collision kernels that
// would be the first contact tick of a run, ~1 ms each in the middle of the simulation).
void preloadReblockKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_touched_flags);
  cudaFuncGetAttributes(&a, k_uf_unite);
  cudaFuncGetAttributes(&a, k_touched_keys);
  cudaFuncGetAttributes(&a, k_cluster_heads);
  cudaFuncGetAttributes(&a, k_cluster_starts);
  cudaFuncGetAttributes(&a, k_cluster_blocks);
  cudaFuncGetAttributes(&a, k_assign_dynamic);
  cudaFuncGetAttributes(&a, k_block_sizes);
  cudaFuncGetAttributes(&a, k_static_membership);
  cudaFuncGetAttributes(&a, k_block_factor);
}

}  // namespace pies
