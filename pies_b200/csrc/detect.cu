// detect.cu — once-per-substep triangle-triangle collision detection.
//
// Replaces reference Solver::_parallelPointTriangleCollisions (Src/Solver.cpp:680-875) and the
// phmap-backed SpatialHash<Triangle> (Include/Pies/SpatialHash.h) with:
//   1. per-triangle swept cell ranges (TriCompRange, exact float semantics, ccd.cuh);
//   2. (cell key, pair index) pairs -> stable radix sort -> cell-start table;
//   3. a self-join narrow phase: a triangle queries exactly the cells it was inserted into
//      (sweptTriRange == TriCompRange except for the 20-cell cap), visiting its cells in key
//      order (= the reference's (dx,dy,dz) order) and each cell's members in ascending index
//      (= bucket order), three corners per candidate;
//   4. hits counted per (triangle, cell) slot of the reference's canonical thread-striped triangle
//      order, scanned, then written, so the output lists are in the reference's order with its
//      multiplicities (SURVEY F7, F8).
// A conservative swept-AABB cull (margin = threshold + slop) skips candidates that cannot
// pass pointTriangleCCD; it never changes the result.
#include "detect.h"

#include "ccd.cuh"

#include <chrono>
#include <cstdio>
#include <cstdlib>

namespace pies {

static inline int gridFor(uint64_t n, int threads) { return (int)((n + threads - 1) / threads); }

// ---- 1. ranges -----------------------------------------------------------------------------
// bbox[0..2] = min cell, bbox[3..5] = max cell (inclusive), bbox[6] = bad-input flag, bbox[7] = hang-guard flag
// `order` (optional) overrides the striping: order[t] = position of local triangle t in the canonical order of the
// GLOBAL scene restricted to the local triangles (slab-partitioned solvers, DESIGN.md section 7).
__device__ __forceinline__ uint32_t canonicalRank(uint32_t t, uint32_t nTri, uint32_t T, const uint32_t* __restrict__ order) {
  if (order) return order[t];
  // thread (t % T) handles t, t+T, ...; per-thread lists are concatenated in thread order (Solver.cpp:714,852-873)
  uint32_t th = t % T, k = t / T;
  uint32_t full = nTri / T, rem = nTri % T;  // threads < rem own full+1 triangles
  return th * full + (th < rem ? th : rem) + k;
}

__global__ void __launch_bounds__(kThreads) k_tri_ranges(uint32_t nTri, uint32_t threadCount, float floorLimit,
                                                         const uint32_t* __restrict__ order,
                                                         const uint32_t* __restrict__ tri,
                                                         const float4* __restrict__ q, const float4* __restrict__ prev,
                                                         int4* __restrict__ triMin, uint4* __restrict__ triRec,
                                                         uint32_t* __restrict__ cnt, uint32_t* __restrict__ cntRank,
                                                         uint32_t* __restrict__ floorRank, float4* __restrict__ aabbLo,
                                                         float4* __restrict__ aabbHi, int* __restrict__ bbox) {
  __shared__ int sb[8];
  if (threadIdx.x < 3) sb[threadIdx.x] = 0x7fffffff;
  else if (threadIdx.x < 6) sb[threadIdx.x] = (int)0x80000000;
  else if (threadIdx.x < 8) sb[threadIdx.x] = 0;
  __syncthreads();
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < nTri) {
    uint32_t a = tri[3 * t], b = tri[3 * t + 1], c = tri[3 * t + 2];
    V3 p0 = v3(q[a]), p1 = v3(q[b]), p2 = v3(q[c]);
    V3 o0 = v3(prev[a]), o1 = v3(prev[b]), o2 = v3(prev[c]);
    int mx, my, mz;
    unsigned lx, ly, lz;
    bool bad;
    ex::triCellRange(p0, p1, p2, o0, o1, o2, mx, my, mz, lx, ly, lz, bad);
    if (bad) sb[6] = 1;
    if (lx > 50u || ly > 50u || lz > 50u) lx = ly = lz = 0;  // TriCompRange cap: not inserted at all
    uint32_t cells = lx * ly * lz;
    // sweptTriRange cap (20 per axis): inserted but queries nothing; a queried range of > 1000 cells
    // trips the reference's hang guard (every cell of the range holds at least this triangle), Solver.cpp:741-745
    if (lx <= 20u && ly <= 20u && lz <= 20u && cells > 1000u) sb[7] = 1;
    triMin[t] = make_int4(mx, my, mz, 0);
    triRec[t] = make_uint4(a, b, c, lx | (ly << 8) | (lz << 16));
    cnt[t] = cells;
    uint32_t rank = canonicalRank(t, nTri, threadCount, order);
    cntRank[rank] = cells;
    // floor test per corner (Solver.cpp:829-834)
    floorRank[rank] = (p0.y < floorLimit ? 1u : 0u) + (p1.y < floorLimit ? 1u : 0u) + (p2.y < floorLimit ? 1u : 0u);
    if (cells) {
      atomicMin(&sb[0], mx); atomicMin(&sb[1], my); atomicMin(&sb[2], mz);
      atomicMax(&sb[3], mx + (int)lx - 1); atomicMax(&sb[4], my + (int)ly - 1); atomicMax(&sb[5], mz + (int)lz - 1);
    }
    aabbLo[t] = make_float4(fminf(fminf(fminf(p0.x, o0.x), fminf(p1.x, o1.x)), fminf(p2.x, o2.x)),
                            fminf(fminf(fminf(p0.y, o0.y), fminf(p1.y, o1.y)), fminf(p2.y, o2.y)),
                            fminf(fminf(fminf(p0.z, o0.z), fminf(p1.z, o1.z)), fminf(p2.z, o2.z)), 0.0f);
    aabbHi[t] = make_float4(fmaxf(fmaxf(fmaxf(p0.x, o0.x), fmaxf(p1.x, o1.x)), fmaxf(p2.x, o2.x)),
                            fmaxf(fmaxf(fmaxf(p0.y, o0.y), fmaxf(p1.y, o1.y)), fmaxf(p2.y, o2.y)),
                            fmaxf(fmaxf(fmaxf(p0.z, o0.z), fmaxf(p1.z, o1.z)), fmaxf(p2.z, o2.z)), 0.0f);
  }
  __syncthreads();
  if (threadIdx.x < 3) { if (sb[threadIdx.x] != 0x7fffffff) atomicMin(bbox + threadIdx.x, sb[threadIdx.x]); }
  else if (threadIdx.x < 6) { if (sb[threadIdx.x] != (int)0x80000000) atomicMax(bbox + threadIdx.x, sb[threadIdx.x]); }
  else if (threadIdx.x < 8) { if (sb[threadIdx.x]) atomicExch(bbox + threadIdx.x, 1); }
}

// floor list in canonical order: scanned floorRank gives each triangle's slot
__global__ void __launch_bounds__(kThreads) k_floor_write(uint32_t nTri, uint32_t threadCount, float floorLimit,
                                                          const uint32_t* __restrict__ order,
                                                          const uint4* __restrict__ triRec, const float4* __restrict__ q,
                                                          const uint32_t* __restrict__ floorRank,
                                                          uint32_t* __restrict__ outFloor) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nTri) return;
  uint32_t rank = canonicalRank(t, nTri, threadCount, order);
  uint32_t beg = floorRank[rank], end = floorRank[rank + 1];
  if (beg == end) return;
  uint4 r = triRec[t];
  uint32_t ids[3] = {r.x, r.y, r.z};
#pragma unroll
  for (int i = 0; i < 3; ++i)
    if (q[ids[i]].y < floorLimit) outFloor[beg++] = ids[i];
}

// ---- 2. pairs ------------------------------------------------------------------------------
struct KeyPack { int minX, minY, minZ; int bitsY, bitsZ; };

// (cell key, triangle) pairs in ascending triangle order, cells of a triangle in (dx,dy,dz) order
__global__ void __launch_bounds__(kThreads) k_emit_pairs(uint32_t nTri, const int4* __restrict__ triMin,
                                                         const uint4* __restrict__ triRec,
                                                         const uint32_t* __restrict__ off, KeyPack kp,
                                                         uint64_t* __restrict__ keys, uint32_t* __restrict__ vals) {
  uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nTri) return;
  uint32_t len = triRec[t].w;
  uint32_t lx = len & 255u, ly = (len >> 8) & 255u, lz = (len >> 16) & 255u;
  if (!(lx * ly * lz)) return;
  int4 m = triMin[t];
  uint32_t i = off[t];
  for (uint32_t dx = 0; dx < lx; ++dx)
    for (uint32_t dy = 0; dy < ly; ++dy)
      for (uint32_t dz = 0; dz < lz; ++dz, ++i) {
        uint64_t kx = (uint64_t)(uint32_t)(m.x + (int)dx - kp.minX);
        uint64_t ky = (uint64_t)(uint32_t)(m.y + (int)dy - kp.minY);
        uint64_t kz = (uint64_t)(uint32_t)(m.z + (int)dz - kp.minZ);
        keys[i] = (kx << (kp.bitsY + kp.bitsZ)) | (ky << kp.bitsZ) | kz;
        vals[i] = t;
      }
}

// ---- 2b. small grids: a direct cell table instead of the radix sort --------------------------------
// When the occupied bounding box has at most 2^22 cells the sorted table is built by counting: every pair takes an
// arrival number from its cell's counter, the counters are scanned into the cell starts, the members are placed at
// start + arrival (arbitrary order) and every pair then finds its rank among its cell's members (ascending triangle
// index = the bucket order of the reference, SURVEY F9).  The cell index of a pair is its key; empty cells are empty ranges.
__global__ void __launch_bounds__(kThreads) k_cell_count(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                         uint32_t* __restrict__ table, uint32_t* __restrict__ arrival) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nPairs) return;
  arrival[i] = atomicAdd(table + (uint32_t)keys[i], 1u);
}

__global__ void __launch_bounds__(kThreads) k_cell_place(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                         const uint32_t* __restrict__ vals, const uint32_t* __restrict__ table,
                                                         const uint32_t* __restrict__ arrival, uint32_t* __restrict__ placed) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nPairs) return;
  placed[table[(uint32_t)keys[i]] + arrival[i]] = vals[i];
}

__global__ void __launch_bounds__(kThreads) k_cell_rank(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                        const uint32_t* __restrict__ vals, const uint32_t* __restrict__ table,
                                                        const uint32_t* __restrict__ placed, uint64_t* __restrict__ outKeys,
                                                        uint32_t* __restrict__ outVals, uint32_t* __restrict__ cellIdx) {
  uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nPairs) return;
  const uint64_t key = keys[i];
  const uint32_t t = vals[i];
  const uint32_t b = table[(uint32_t)key], e = table[(uint32_t)key + 1];
  uint32_t rank = 0;
  for (uint32_t k = b; k < e; ++k) rank += placed[k] < t ? 1u : 0u;
  outKeys[b + rank] = key;
  outVals[b + rank] = t;
  cellIdx[b + rank] = (uint32_t)key;
}

// ---- 3. cell-start table -------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads) k_mark_heads(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                         uint32_t* __restrict__ heads) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j > nPairs) return;
  heads[j] = (j < nPairs && (j == 0 || keys[j] != keys[j - 1])) ? 1u : 0u;
}

// cellIdx (in place of the scanned heads) and cellStart
__global__ void __launch_bounds__(kThreads) k_cell_starts(uint64_t nPairs, const uint64_t* __restrict__ keys,
                                                          uint32_t* __restrict__ headScan /* -> cellIdx */,
                                                          uint32_t* __restrict__ cellStart) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nPairs) return;
  bool head = (j == 0 || keys[j] != keys[j - 1]);
  uint32_t idx = headScan[j] + (head ? 1u : 0u) - 1u;
  if (head) cellStart[idx] = (uint32_t)j;
  if (j == nPairs - 1) cellStart[idx + 1] = (uint32_t)nPairs;
  headScan[j] = idx;
}

// ---- 4. narrow phase ------------------------------------------------------------------------
// 4a. candidate filter: one thread per (cell, member) pair of the sorted table.  The member triangle is
// compared with every triangle of that cell — what the reference's worker does when it visits this bucket
// for this triangle — but only with the cheap tests: shared node, then swept corner box against the other
// triangle's swept box (conservative: a pair that fails it cannot pass pointTriangleCCD).  Neighbouring
// threads sit in the same cell, so the member loop reads the same records in every lane (broadcast) while
// each lane keeps its own triangle in registers.  The member loop runs ONCE: it counts the pair's candidates
// and remembers which members produced any (a 64-bit mask; cells with more members redo the loop), the warp
// reserves one contiguous chunk of the candidate buffer for all its pairs, and every thread writes its run
// there.  The chunk order is arbitrary; the runs are found again through pairRun[j].
// 4b. CCD: one thread per candidate (point, triangle), in the cell-sorted order of the candidate buffer
// (neighbouring candidates share nodes and triangles): the expensive swept test runs exactly once per
// candidate, fully convergent.
// 4c. hits in the reference's order: the hits of pair (t, k-th cell of t) are counted into slot
// rankOff[rank(t)] + k (thread-striped triangle order, cells in (dx,dy,dz) order); after a scan over the
// slots the same kernel writes them (members ascending, corners 0..2 inside a run) — the output lists come
// out in the reference's order with its multiplicities (SURVEY F7, F8) without atomics on the ordering path.
struct NarrowParams {
  uint32_t nTri, threadCount;
  float threshold;
  float cullMargin;
  const uint32_t* order;
};

__global__ void __launch_bounds__(kThreads) k_pair_filter(NarrowParams np, KeyPack kp, uint64_t nPairs,
                                                          const uint64_t* __restrict__ keys,
                                                          const uint32_t* __restrict__ memberTri,
                                                          const uint32_t* __restrict__ cellIdx,
                                                          const uint32_t* __restrict__ cellStart,
                                                          const uint4* __restrict__ triRec, const int4* __restrict__ triMin,
                                                          const float4* __restrict__ aabbLo, const float4* __restrict__ aabbHi,
                                                          const float4* __restrict__ q, const float4* __restrict__ prev,
                                                          const uint32_t* __restrict__ rankOff,
                                                          uint2* __restrict__ pairRun /* (first candidate, count) */,
                                                          uint32_t* __restrict__ pairSlot /* canonical slot */,
                                                          uint2* __restrict__ cand, uint32_t candCap,
                                                          uint32_t* __restrict__ candTotal, int* __restrict__ failFlag) {
  const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = j < nPairs;
  uint32_t total = 0, s = 0, e = 0, slot = 0;
  uint64_t mask = 0;
  uint32_t ia[3] = {0, 0, 0};
  float cLo[3][3], cHi[3][3];
  if (live) {
    uint32_t t = memberTri[j];
    uint4 rec = triRec[t];
    uint32_t lx = rec.w & 255u, ly = (rec.w >> 8) & 255u, lz = (rec.w >> 16) & 255u;
    // slot of (t, this cell) in the canonical order
    uint64_t key = keys[j];
    int4 mn = triMin[t];
    uint32_t dz = (uint32_t)((int)(key & ((1ull << kp.bitsZ) - 1ull)) + kp.minZ - mn.z);
    uint32_t dy = (uint32_t)((int)((key >> kp.bitsZ) & ((1ull << kp.bitsY) - 1ull)) + kp.minY - mn.y);
    uint32_t dx = (uint32_t)((int)(key >> (kp.bitsY + kp.bitsZ)) + kp.minX - mn.x);
    slot = rankOff[canonicalRank(t, np.nTri, np.threadCount, np.order)] + (dx * ly + dy) * lz + dz;
    if (lx <= 20u && ly <= 20u && lz <= 20u) {  // sweptTriRange cap: beyond it the triangle is inserted but queries nothing
      uint32_t cidx = cellIdx[j];
      s = cellStart[cidx]; e = cellStart[cidx + 1];
      if (e - s > 1000u) atomicExch(failFlag, 1);  // hang guard, Solver.cpp:751-755
      ia[0] = rec.x; ia[1] = rec.y; ia[2] = rec.z;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
        float4 p = q[ia[i]], o = prev[ia[i]];
        cLo[i][0] = fminf(p.x, o.x) - np.cullMargin; cHi[i][0] = fmaxf(p.x, o.x) + np.cullMargin;
        cLo[i][1] = fminf(p.y, o.y) - np.cullMargin; cHi[i][1] = fmaxf(p.y, o.y) + np.cullMargin;
        cLo[i][2] = fminf(p.z, o.z) - np.cullMargin; cHi[i][2] = fmaxf(p.z, o.z) + np.cullMargin;
      }
      // union of the three corner boxes: one test rejects most members
      float uLo[3], uHi[3];
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        uLo[c] = fminf(cLo[0][c], fminf(cLo[1][c], cLo[2][c]));
        uHi[c] = fmaxf(cHi[0][c], fmaxf(cHi[1][c], cHi[2][c]));
      }
      // (a software-pipelined variant — member records one iteration ahead — was measured slower, r02t: 364 vs 330 us;
      // the registers it takes cost more occupancy than the overlap wins)
      uint32_t oNext = memberTri[s];
      for (uint32_t m = s; m < e; ++m) {
        const uint32_t o = oNext;
        if (m + 1 < e) oNext = memberTri[m + 1];
        const uint4 ro = triRec[o];
        const float4 lo = aabbLo[o], hi = aabbHi[o];  // issued with the record: the three loads only depend on o
        bool common = false;
#pragma unroll
        for (int i = 0; i < 3; ++i) common |= (ia[i] == ro.x) | (ia[i] == ro.y) | (ia[i] == ro.z);
        if (common) continue;
        if (!(uLo[0] <= hi.x && uHi[0] >= lo.x && uLo[1] <= hi.y && uHi[1] >= lo.y && uLo[2] <= hi.z && uHi[2] >= lo.z)) continue;
        uint32_t c = 0;
#pragma unroll
        for (int i = 0; i < 3; ++i)
          c += (cLo[i][0] <= hi.x && cHi[i][0] >= lo.x && cLo[i][1] <= hi.y && cHi[i][1] >= lo.y && cLo[i][2] <= hi.z &&
                cHi[i][2] >= lo.z) ? 1u : 0u;
        if (c) { total += c; if (m - s < 64u) mask |= 1ull << (m - s); }
      }
    }
  }
  // exclusive scan of the totals over the warp, one reservation per warp (no CTA barrier: the member loops of a CTA's
  // warps differ widely in length)
  const int lane = threadIdx.x & 31;
  uint32_t inc = total;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += v; }
  uint32_t chunkBase = 0;
  if (lane == 31 && inc) chunkBase = atomicAdd(candTotal, inc);
  chunkBase = __shfl_sync(0xffffffffu, chunkBase, 31);
  if (!live) return;
  uint32_t pos = chunkBase + inc - total;
  pairRun[j] = make_uint2(pos, total);
  pairSlot[j] = slot;
  if (!total) return;
  const bool wide = e - s > 64u;
  for (uint32_t m = s; m < e; ++m) {
    if (!wide) {
      if (!mask) break;
      uint32_t b = (uint32_t)__ffsll((long long)mask) - 1u;
      mask &= mask - 1ull;
      m = s + b;
    }
    uint32_t o = memberTri[m];
    if (wide) {
      uint4 ro = triRec[o];
      bool common = false;
#pragma unroll
      for (int i = 0; i < 3; ++i) common |= (ia[i] == ro.x) | (ia[i] == ro.y) | (ia[i] == ro.z);
      if (common) continue;
    }
    float4 lo = aabbLo[o], hi = aabbHi[o];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
      bool ov = cLo[i][0] <= hi.x && cHi[i][0] >= lo.x && cLo[i][1] <= hi.y && cHi[i][1] >= lo.y &&
                cLo[i][2] <= hi.z && cHi[i][2] >= lo.z;
      if (ov) {
        if (pos < candCap) cand[pos] = make_uint2(ia[i], o);
        ++pos;
      }
    }
  }
}

__global__ void __launch_bounds__(128) k_ccd(const uint32_t* __restrict__ nCandPtr, uint32_t candCap,
                                             const uint2* __restrict__ cand, const uint4* __restrict__ triRec,
                                             const float4* __restrict__ q, const float4* __restrict__ prev,
                                             float threshold, uint8_t* __restrict__ hit) {
  uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
  uint32_t nCand = min(*nCandPtr, candCap);
  if (k >= nCand) return;
  uint2 cd = cand[k];
  uint4 ro = triRec[cd.y];
  V3 pa = v3(q[cd.x]), oa = v3(prev[cd.x]);
  V3 pb = v3(q[ro.x]), pc = v3(q[ro.y]), pd = v3(q[ro.z]);
  V3 ob = v3(prev[ro.x]), oc = v3(prev[ro.y]), od = v3(prev[ro.z]);
  float tt;
  bool h = ex::pointTriangleCCD(ex::sub(oa, ob), ex::sub(oc, ob), ex::sub(od, ob), ex::sub(pa, pb), ex::sub(pc, pb),
                                ex::sub(pd, pb), threshold, tt);
  hit[k] = h ? 1 : 0;
}

// WRITE == false: hits of every pair into its canonical slot; WRITE == true (after the scan over the slots): the hits
// themselves, in run order.
template <bool WRITE>
__global__ void __launch_bounds__(kThreads) k_pair_hits(uint64_t nPairs, const uint2* __restrict__ pairRun,
                                                        const uint32_t* __restrict__ pairSlot, uint32_t candCap,
                                                        const uint8_t* __restrict__ hit, uint32_t* __restrict__ hitCount,
                                                        const uint2* __restrict__ cand, const uint4* __restrict__ triRec,
                                                        uint4* __restrict__ outTri, uint32_t* __restrict__ outOther) {
  uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= nPairs) return;
  if (!WRITE && j == 0) hitCount[nPairs] = 0;
  const uint2 run = pairRun[j];
  const uint32_t slot = pairSlot[j];
  const uint32_t end = min(run.x + run.y, candCap);
  if (!WRITE) {
    uint32_t c = 0;
    for (uint32_t k = run.x; k < end; ++k) c += hit[k];
    hitCount[slot] = c;
  } else {
    uint32_t pos = hitCount[slot];
    if (hitCount[slot + 1] == pos) return;
    for (uint32_t k = run.x; k < end; ++k) {
      if (!hit[k]) continue;
      uint2 cd = cand[k];
      uint4 ro = triRec[cd.y];
      outTri[pos] = make_uint4(cd.x, ro.x, ro.y, ro.z);
      outOther[pos] = cd.y;
      ++pos;
    }
  }
}

// ---- 5. node -> incident entries --------------------------------------------------------------
// A counting sort by node: every (entry, slot) item takes an arrival number from its node's counter, the counters are
// scanned into the CSR offsets and the items are placed at offset + arrival (arbitrary order inside a node).  Whatever
// needs the node's list in ascending order then ranks the item inside its (short) list — one thread per item, the list
// read from L1.  The result equals a stable sort by node of the items in index order, without radix passes.
__device__ __forceinline__ uint32_t comp(const uint4& v, uint32_t s) { return s == 0u ? v.x : (s == 1u ? v.y : (s == 2u ? v.z : v.w)); }

__global__ void __launch_bounds__(kThreads) k_inc_count(uint32_t nEntries, const uint32_t* __restrict__ nEntriesDev,
                                                        const uint4* __restrict__ entries, uint32_t* __restrict__ incCount,
                                                        uint32_t* __restrict__ arrival) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nEntries || (nEntriesDev && e >= *nEntriesDev)) return;
  uint4 v = entries[e];
  uint32_t ids[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int s = 0; s < 4; ++s) arrival[4ull * e + s] = atomicAdd(incCount + ids[s], 1u);
}

// pointTri (optional): the triangle of the entry for its point item (slot 0), ~0 for the corner items
__global__ void __launch_bounds__(kThreads) k_inc_place(uint32_t nEntries, const uint32_t* __restrict__ nEntriesDev,
                                                        const uint4* __restrict__ entries, const uint32_t* __restrict__ incPtr,
                                                        const uint32_t* __restrict__ arrival, uint32_t* __restrict__ placed,
                                                        const uint32_t* __restrict__ otherTri, uint32_t* __restrict__ pointTri) {
  uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nEntries || (nEntriesDev && e >= *nEntriesDev)) return;
  uint4 v = entries[e];
  uint32_t ids[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int s = 0; s < 4; ++s) {
    const uint32_t at = incPtr[ids[s]] + arrival[4ull * e + s];
    placed[at] = 4u * e + s;
    if (pointTri) pointTri[at] = s == 0 ? otherTri[e] : 0xffffffffu;
  }
}

// One thread per item of the FULL contact list (every copy):
//  * ticket = its position in the node's list ordered by entry — the ordered Gauss-Seidel sweeps (contact.cu) run an
//    entry once each of its four nodes has seen `ticket` earlier entries;
//  * distinct contacts: the reference's list holds the same (point, triangle) once per shared cell and per triangle the
//    point is a corner of (SURVEY F7); the ordered sweeps need every copy, but the collision MATRIX and the right-hand
//    side only need each distinct contact with its multiplicity.  Among a node's point items the first copy of each
//    triangle is the head: it keeps the number of copies and counts into uCount[node].
__global__ void __launch_bounds__(kThreads) k_item_contacts(uint64_t nInc, const uint4* __restrict__ entries,
                                                            const uint32_t* __restrict__ incPtr,
                                                            const uint32_t* __restrict__ placed,
                                                            const uint32_t* __restrict__ pointTri, uint32_t* __restrict__ ticket,
                                                            uint32_t* __restrict__ headTri, uint32_t* __restrict__ uMult,
                                                            uint32_t* __restrict__ uCount) {
  const uint64_t at = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (at >= nInc) return;
  const uint32_t v = placed[at];
  const uint32_t node = comp(entries[v >> 2], v & 3u);
  const uint32_t b = incPtr[node], k = incPtr[node + 1] - b;
  const uint32_t tri = pointTri[at];
  uint32_t rank = 0, mult = 0, earlier = 0;
  if (tri == 0xffffffffu) {
    for (uint32_t j = 0; j < k; ++j) rank += placed[b + j] < v ? 1u : 0u;
  } else {
    for (uint32_t j = 0; j < k; ++j) {
      const uint32_t vj = placed[b + j];
      const bool same = pointTri[b + j] == tri, less = vj < v;
      rank += less ? 1u : 0u;
      mult += same ? 1u : 0u;
      earlier += same && less ? 1u : 0u;
    }
  }
  ticket[v] = rank;
  const bool head = tri != 0xffffffffu && earlier == 0u;
  headTri[at] = head ? tri : 0xffffffffu;
  uMult[at] = mult;
  if (head) atomicAdd(uCount + node, 1u);
}

// Distinct contacts in (point, triangle) order with their weights (a head's rank among its node's heads = number of
// smaller triangles), and the arrival numbers for THEIR incidence table.
__global__ void __launch_bounds__(kThreads) k_uniq_write(uint64_t nInc, const uint32_t* __restrict__ placed,
                                                         const uint32_t* __restrict__ headTri,
                                                         const uint32_t* __restrict__ uMult,
                                                         const uint32_t* __restrict__ incPtr,
                                                         const uint32_t* __restrict__ uStart /* scanned uCount */,
                                                         const uint4* __restrict__ entries, uint4* __restrict__ uTri,
                                                         float* __restrict__ uW, uint32_t* __restrict__ uIncCount,
                                                         uint32_t* __restrict__ uArrival) {
  const uint64_t at = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (at >= nInc) return;
  const uint32_t tri = headTri[at];
  if (tri == 0xffffffffu) return;
  const uint4 e = entries[placed[at] >> 2];
  const uint32_t b = incPtr[e.x], k = incPtr[e.x + 1] - b;
  uint32_t r = 0;
  for (uint32_t j = 0; j < k; ++j) r += headTri[b + j] < tri ? 1u : 0u;
  const uint32_t u = uStart[e.x] + r;
  uTri[u] = e;
  uW[u] = 10000.0f * (float)uMult[at];  // copies * PointTriangleCollisionConstraint::w (exact in fp32)
  uint32_t ids[4] = {e.x, e.y, e.z, e.w};
#pragma unroll
  for (int s = 0; s < 4; ++s) uArrival[4ull * u + s] = atomicAdd(uIncCount + ids[s], 1u);
}

// One thread per placed item: to its rank inside the node's list (ascending values).
__global__ void __launch_bounds__(kThreads) k_item_sort(uint64_t nItemsBound, const uint32_t* __restrict__ nEntriesDev,
                                                        const uint4* __restrict__ entries, const uint32_t* __restrict__ ptr,
                                                        const uint32_t* __restrict__ placed, uint32_t* __restrict__ sorted) {
  const uint64_t at = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (at >= nItemsBound || at >= 4ull * *nEntriesDev) return;
  const uint32_t v = placed[at];
  const uint32_t node = comp(entries[v >> 2], v & 3u);
  const uint32_t b = ptr[node], k = ptr[node + 1] - b;
  uint32_t rank = 0;
  for (uint32_t j = 0; j < k; ++j) rank += placed[b + j] < v ? 1u : 0u;
  sorted[b + rank] = v;
}

__global__ void __launch_bounds__(kThreads) k_floor_mult(uint32_t nFloor, const uint32_t* __restrict__ nodes,
                                                         uint32_t* __restrict__ mult) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < nFloor) atomicAdd(mult + nodes[i], 1u);
}

__global__ void __launch_bounds__(kThreads) k_floor_weight(uint32_t n, const uint32_t* __restrict__ mult,
                                                           float* __restrict__ w) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float acc = 0.0f;
  for (uint32_t k = 0; k < mult[i]; ++k) acc += 10000.0f;  // StaticCollisionConstraint::w, coeffRef += per duplicate
  w[i] = acc;
}

// ---- 7. the collision matrix in streamable form ----------------------------------------------------
// Off-diagonal entries per node (to be scanned): a contact contributes three to its point row and one to each
// corner row (A^T A = [[3,-1,-1,-1],[-1,1,0,0],[-1,0,1,0],[-1,0,0,1]], CollisionConstraint.cpp:74-83).
__global__ void __launch_bounds__(kThreads) k_ccsr_count(uint32_t n, const uint32_t* __restrict__ uIncPtr,
                                                         const uint32_t* __restrict__ uInc, uint32_t* __restrict__ cPtr) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > n) return;
  uint32_t cnt = 0;
  if (i < n)
    for (uint32_t k = uIncPtr[i]; k < uIncPtr[i + 1]; ++k) cnt += (uInc[k] & 3u) == 0u ? 3u : 1u;
  cPtr[i] = cnt;
}

// Entries in the node's incidence order (contacts ascending), diagonal = contact terms then the floor weight.
__global__ void __launch_bounds__(kThreads) k_ccsr_fill(uint32_t n, const uint32_t* __restrict__ uIncPtr,
                                                        const uint32_t* __restrict__ uInc, const uint4* __restrict__ uTri,
                                                        const float* __restrict__ uW, const uint32_t* __restrict__ cPtr,
                                                        const float* __restrict__ floorW, int* __restrict__ cCol,
                                                        float* __restrict__ cVal, float* __restrict__ cDiag) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float diag = 0.0f;
  if (uIncPtr) {
    uint32_t o = cPtr[i];
    for (uint32_t k = uIncPtr[i]; k < uIncPtr[i + 1]; ++k) {
      const uint32_t v = uInc[k];
      const uint4 e = uTri[v >> 2];
      const float wgt = uW[v >> 2];
      if ((v & 3u) == 0u) {
        diag += 3.0f * wgt;
        cCol[o] = (int)e.y; cCol[o + 1] = (int)e.z; cCol[o + 2] = (int)e.w;
        cVal[o] = -wgt; cVal[o + 1] = -wgt; cVal[o + 2] = -wgt;
        o += 3;
      } else {
        diag += wgt;
        cCol[o] = (int)e.x; cVal[o] = -wgt;
        ++o;
      }
    }
  }
  if (floorW) diag += floorW[i];
  cDiag[i] = diag;
}

__global__ void k_init_bbox(int* bbox) {
  bbox[0] = bbox[1] = bbox[2] = 0x7fffffff;
  bbox[3] = bbox[4] = bbox[5] = (int)0x80000000;
  bbox[6] = 0; bbox[7] = 0;
}

static int bitsFor(int64_t span) {  // bits to hold values 0..span
  int b = 1;
  while ((int64_t(1) << b) <= span) ++b;
  return b;
}

#define DCHECK(expr)                                                    \
  do {                                                                  \
    cudaError_t _e = (expr);                                            \
    if (_e != cudaSuccess) { w.lastError = _e; return -1; }             \
  } while (0)

int detectTriangles(DetectWork& w, cudaStream_t s, const DetectInput& in, ContactLists& out, int* launches) {
  int L = 0;
  // diagnostics: host time stamps around the three synchronisations (PIES_B200_DETECT_TRACE)
  static const bool traceOn = std::getenv("PIES_B200_DETECT_TRACE") != nullptr;
  double stamp[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  auto mark = [&](int k) { if (traceOn) stamp[k] = std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
  mark(0);
  const uint32_t nTri = in.nTri, n = in.nNodes;
  const uint32_t T = in.threadCount ? in.threadCount : 1u;
  const float floorLimit = in.floorLimit;
  out.nTri = out.nFloor = 0;
  w.nPairs = 0; w.nCells = 0; w.nUnique = 0; w.failed = false; w.badInput = false;
  DCHECK(w.incPtr.reserve(n + 2));
  DCHECK(w.floorMult.reserve(n + 1));
  DCHECK(w.floorW.reserve(n + 1));
  DCHECK(w.nodeDone.reserve(n + 1));
  out.floorW = w.floorW.p; out.floorMult = w.floorMult.p; out.nodeDone = w.nodeDone.p;
  const uint32_t nCol = in.colliders.n;
  // static colliders: every node's mask, their weights after the floor's (floorW), published with the lists
  auto colliderPass = [&](bool haveFloor) {
    if (!nCol) return;
    L += launchColliderDetect(s, n, in.colliders, in.q, in.thickness, haveFloor, in.colMask, w.floorW.p);
    out.nCollide = nCol; out.colMask = in.colMask;
  };
  const uint32_t nDrag = in.drags.n;
  // drag targets: their weights after the floor's and the colliders' (floorW is zeroed first when neither wrote it this
  // substep), and w g into msn, in one launch
  auto dragPass = [&](bool haveFloorW) -> cudaError_t {
    if (!nDrag) return cudaSuccess;
    if (!haveFloorW) {
      const cudaError_t e = cudaMemsetAsync(w.floorW.p, 0, (size_t)n * sizeof(float), s);
      if (e != cudaSuccess) return e;
    }
    L += launchDragTerms(s, in.drags, w.floorW.p, in.msn);
    out.nDrag = nDrag;
    return cudaSuccess;
  };
  if (!nTri) {
    if ((nCol || nDrag) && n) {  // no triangles (bare nodes, ropes): only the colliders' and drags' diagonal
      colliderPass(false);
      DCHECK(dragPass(nCol != 0));
      DCHECK(w.cDiag.reserve(n + 1));
      k_ccsr_fill<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, nullptr, nullptr, nullptr, nullptr, nullptr, w.floorW.p, nullptr,
                                                           nullptr, w.cDiag.p); ++L;
      out.cDiag = w.cDiag.p;
    }
    if (launches) *launches += L;
    return 0;
  }
  DCHECK(w.triMin.reserve(nTri)); DCHECK(w.triRec.reserve(nTri)); DCHECK(w.cnt.reserve(nTri + 2));
  DCHECK(w.cntRank.reserve(nTri + 2)); DCHECK(w.floorRank.reserve(nTri + 2));
  DCHECK(w.aabbLo.reserve(nTri)); DCHECK(w.aabbHi.reserve(nTri));
  DCHECK(w.bbox.reserve(12));
  DCHECK(w.scanScratch.reserve(scanScratchElems(std::max<uint64_t>(nTri + 2, w.scanCap))));
  k_init_bbox<<<1, 1, 0, s>>>(w.bbox.p); ++L;
  DCHECK(cudaMemsetAsync(w.cnt.p + nTri, 0, 2 * sizeof(uint32_t), s));
  DCHECK(cudaMemsetAsync(w.cntRank.p + nTri, 0, 2 * sizeof(uint32_t), s));
  DCHECK(cudaMemsetAsync(w.floorRank.p + nTri, 0, 2 * sizeof(uint32_t), s));
  k_tri_ranges<<<gridFor(nTri, kThreads), kThreads, 0, s>>>(nTri, T, floorLimit, in.order, in.tri, in.q, in.prev, w.triMin.p, w.triRec.p,
                                                           w.cnt.p, w.cntRank.p, w.floorRank.p, w.aabbLo.p, w.aabbHi.p,
                                                           w.bbox.p); ++L;
  L += launchExclusiveScan(s, w.cnt.p, nTri + 1, w.scanScratch.p);
  L += launchExclusiveScan(s, w.cntRank.p, nTri + 1, w.scanScratch.p);
  L += launchExclusiveScan(s, w.floorRank.p, nTri + 1, w.scanScratch.p);
  DCHECK(cudaMemcpyAsync(w.host, w.bbox.p, 8 * sizeof(int), cudaMemcpyDeviceToHost, s));
  DCHECK(cudaMemcpyAsync(w.host + 8, w.cnt.p + nTri, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  DCHECK(cudaMemcpyAsync(w.host + 11, w.floorRank.p + nTri, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
  mark(1);
  DCHECK(cudaStreamSynchronize(s));
  mark(2);
  if (w.host[6]) { w.badInput = true; return 0; }
  if (w.host[7]) { w.failed = true; if (launches) *launches += L; return 0; }  // reference latches _simFailed, lists stay empty
  uint64_t nPairs = (uint32_t)w.host[8];
  uint32_t nFloor = (uint32_t)w.host[11];
  w.nPairs = nPairs;
  NarrowParams np{nTri, T, in.threshold, in.threshold + 1e-3f, in.order};
  uint32_t nHit = 0;
  if (nPairs) {
    KeyPack kp{w.host[0], w.host[1], w.host[2], 0, 0};
    int bx = bitsFor((int64_t)w.host[3] - w.host[0]), by = bitsFor((int64_t)w.host[4] - w.host[1]),
        bz = bitsFor((int64_t)w.host[5] - w.host[2]);
    kp.bitsY = by; kp.bitsZ = bz;
    if (bx + by + bz > 63) { w.badInput = true; return 0; }
    w.keyPack[0] = kp.minX; w.keyPack[1] = kp.minY; w.keyPack[2] = kp.minZ; w.keyPack[3] = by; w.keyPack[4] = bz;
    DCHECK(w.keys.reserve(nPairs)); DCHECK(w.tmpKeys.reserve(nPairs));
    DCHECK(w.vals.reserve(nPairs)); DCHECK(w.tmpVals.reserve(nPairs));
    DCHECK(w.heads.reserve(nPairs + 2)); DCHECK(w.cellStart.reserve(nPairs + 2)); DCHECK(w.hitCount.reserve(nPairs + 2));
    DCHECK(w.sortHist.reserve(sortHistBytes(nPairs) / 4 + 4));
    w.scanCap = std::max<uint64_t>(w.scanCap, nPairs + 2);
    DCHECK(w.scanScratch.reserve(scanScratchElems(w.scanCap)));
    static const bool noCellTable = std::getenv("PIES_B200_NO_CELL_TABLE") != nullptr;   // A/B switch: always radix-sort
    const int keyBits = bx + by + bz;
    const bool direct = keyBits <= 22 && !noCellTable;
    const uint32_t* cellStart = nullptr;
    if (direct) {
      const size_t cells = (size_t)1 << keyBits;
      DCHECK(w.cellTable.reserve(cells + 2)); DCHECK(w.arrivalP.reserve(nPairs)); DCHECK(w.placedP.reserve(nPairs));
      w.scanCap = std::max<uint64_t>(w.scanCap, cells + 2);
      DCHECK(w.scanScratch.reserve(scanScratchElems(w.scanCap)));
      DCHECK(cudaMemsetAsync(w.cellTable.p, 0, (cells + 2) * sizeof(uint32_t), s));
      k_emit_pairs<<<gridFor(nTri, kThreads), kThreads, 0, s>>>(nTri, w.triMin.p, w.triRec.p, w.cnt.p, kp, w.tmpKeys.p, w.tmpVals.p); ++L;
      k_cell_count<<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.tmpKeys.p, w.cellTable.p, w.arrivalP.p); ++L;
      L += launchExclusiveScan(s, w.cellTable.p, cells + 1, w.scanScratch.p);
      k_cell_place<<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.tmpKeys.p, w.tmpVals.p, w.cellTable.p, w.arrivalP.p,
                                                                 w.placedP.p); ++L;
      k_cell_rank<<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.tmpKeys.p, w.tmpVals.p, w.cellTable.p, w.placedP.p,
                                                                w.keys.p, w.vals.p, w.heads.p); ++L;
      w.host[9] = 0;
      cellStart = w.cellTable.p;
    } else {
      k_emit_pairs<<<gridFor(nTri, kThreads), kThreads, 0, s>>>(nTri, w.triMin.p, w.triRec.p, w.cnt.p, kp, w.keys.p, w.vals.p); ++L;
      L += launchSortPairs(s, nPairs, w.keys.p, w.vals.p, w.tmpKeys.p, w.tmpVals.p, w.sortHist.p, keyBits);
      k_mark_heads<<<gridFor(nPairs + 1, kThreads), kThreads, 0, s>>>(nPairs, w.keys.p, w.heads.p); ++L;
      L += launchExclusiveScan(s, w.heads.p, nPairs + 1, w.scanScratch.p);
      DCHECK(cudaMemcpyAsync(w.host + 9, w.heads.p + nPairs, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      k_cell_starts<<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.keys.p, w.heads.p, w.cellStart.p); ++L;
      cellStart = w.cellStart.p;
    }
    // candidate filter (one pass, capacity from the previous substep; redone if it overflows), CCD, hits per slot, scan
    DCHECK(w.pairRun.reserve(nPairs)); DCHECK(w.pairSlot.reserve(nPairs));
    uint32_t nCand = 0, cap = 0;
    for (int attempt = 0; attempt < 2; ++attempt) {
      cap = std::max<uint32_t>(w.candCap, 1u << 16);
      DCHECK(w.cand.reserve(cap)); DCHECK(w.candHit.reserve((size_t)cap + 16));
      DCHECK(cudaMemsetAsync(w.bbox.p + 8, 0, sizeof(int), s));
      k_pair_filter<<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(np, kp, nPairs, w.keys.p, w.vals.p, w.heads.p, cellStart,
                                                                 w.triRec.p, w.triMin.p, w.aabbLo.p, w.aabbHi.p, in.q, in.prev,
                                                                 w.cntRank.p, w.pairRun.p, w.pairSlot.p, w.cand.p, cap,
                                                                 (uint32_t*)(w.bbox.p + 8), w.bbox.p + 7); ++L;
      k_ccd<<<gridFor(cap, 128), 128, 0, s>>>((const uint32_t*)(w.bbox.p + 8), cap, w.cand.p, w.triRec.p, in.q, in.prev,
                                             in.threshold, w.candHit.p); ++L;
      k_pair_hits<false><<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.pairRun.p, w.pairSlot.p, cap, w.candHit.p,
                                                                      w.hitCount.p, nullptr, nullptr, nullptr, nullptr); ++L;
      L += launchExclusiveScan(s, w.hitCount.p, nPairs + 1, w.scanScratch.p);
      DCHECK(cudaMemcpyAsync(w.host + 14, w.bbox.p + 8, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      DCHECK(cudaMemcpyAsync(w.host + 12, w.bbox.p + 7, sizeof(int), cudaMemcpyDeviceToHost, s));
      DCHECK(cudaMemcpyAsync(w.host + 10, w.hitCount.p + nPairs, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      mark(3);
      DCHECK(cudaStreamSynchronize(s));
      mark(4);
      nCand = (uint32_t)w.host[14];
      if (nCand <= cap) break;
      if (attempt == 1) { w.lastError = cudaErrorUnknown; return -1; }  // the count cannot change between attempts
      w.candCap = nCand + nCand / 2;  // overflow: the list was truncated, redo with room
    }
    w.candCap = std::max<uint32_t>(w.candCap, nCand + nCand / 4 + 1024);
    w.nCells = (uint32_t)w.host[9];
    if (w.host[12]) { w.failed = true; if (launches) *launches += L; return 0; }
    nHit = (uint32_t)w.host[10];
    DCHECK(w.triList.reserve(nHit + 1)); DCHECK(w.otherTri.reserve(nHit + 1));
    if (nHit) {
      k_pair_hits<true><<<gridFor(nPairs, kThreads), kThreads, 0, s>>>(nPairs, w.pairRun.p, w.pairSlot.p, cap, w.candHit.p,
                                                                     w.hitCount.p, w.cand.p, w.triRec.p, w.triList.p,
                                                                     w.otherTri.p); ++L;
    }
  }
  DCHECK(w.floorList.reserve(nFloor + 1));
  if (nFloor) {
    k_floor_write<<<gridFor(nTri, kThreads), kThreads, 0, s>>>(nTri, T, floorLimit, in.order, w.triRec.p, in.q, w.floorRank.p,
                                                              w.floorList.p); ++L;
  }
  out.tri = w.triList.p; out.floorNode = w.floorList.p; out.nTri = nHit; out.nFloor = nFloor;
  // incidence CSR + tickets + floor multiplicities
  if (nHit) {
    const uint64_t nInc = 4ull * nHit;
    DCHECK(cudaMemsetAsync(w.incPtr.p, 0, (n + 2) * sizeof(uint32_t), s));
    DCHECK(w.arrival.reserve(nInc)); DCHECK(w.placed.reserve(nInc)); DCHECK(w.ticket.reserve(nInc));
    DCHECK(w.pointTri.reserve(nInc)); DCHECK(w.headTri.reserve(nInc)); DCHECK(w.uMult.reserve(nInc));
    DCHECK(w.uStart.reserve(n + 2)); DCHECK(w.uIncPtr.reserve(n + 2));
    DCHECK(w.uTri.reserve(nHit)); DCHECK(w.uW.reserve(nHit)); DCHECK(w.uInc.reserve(nInc));
    w.scanCap = std::max<uint64_t>(w.scanCap, (uint64_t)n + 2);
    DCHECK(w.scanScratch.reserve(scanScratchElems(w.scanCap)));
    k_inc_count<<<gridFor(nHit, kThreads), kThreads, 0, s>>>(nHit, nullptr, w.triList.p, w.incPtr.p, w.arrival.p); ++L;
    L += launchExclusiveScan(s, w.incPtr.p, n + 1, w.scanScratch.p);
    k_inc_place<<<gridFor(nHit, kThreads), kThreads, 0, s>>>(nHit, nullptr, w.triList.p, w.incPtr.p, w.arrival.p, w.placed.p,
                                                            w.otherTri.p, w.pointTri.p); ++L;
    DCHECK(cudaMemsetAsync(w.uStart.p, 0, (n + 2) * sizeof(uint32_t), s));
    k_item_contacts<<<gridFor(nInc, kThreads), kThreads, 0, s>>>(nInc, w.triList.p, w.incPtr.p, w.placed.p, w.pointTri.p,
                                                                w.ticket.p, w.headTri.p, w.uMult.p, w.uStart.p); ++L;
    out.ticket = reinterpret_cast<uint4*>(w.ticket.p);
    // distinct contacts with multiplicity (sorted by (point, triangle)), then their node incidence table; the host
    // only learns their number at the end (everything is sized by the full list)
    L += launchExclusiveScan(s, w.uStart.p, n + 1, w.scanScratch.p);
    DCHECK(cudaMemcpyAsync(w.host + 13, w.uStart.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
    DCHECK(cudaMemsetAsync(w.uIncPtr.p, 0, (n + 2) * sizeof(uint32_t), s));
    k_uniq_write<<<gridFor(nInc, kThreads), kThreads, 0, s>>>(nInc, w.placed.p, w.headTri.p, w.uMult.p, w.incPtr.p, w.uStart.p,
                                                             w.triList.p, w.uTri.p, w.uW.p, w.uIncPtr.p, w.arrival.p); ++L;
    L += launchExclusiveScan(s, w.uIncPtr.p, n + 1, w.scanScratch.p);
    k_inc_place<<<gridFor(nHit, kThreads), kThreads, 0, s>>>(nHit, w.uStart.p + n, w.uTri.p, w.uIncPtr.p, w.arrival.p,
                                                            w.placed.p, nullptr, nullptr); ++L;
    k_item_sort<<<gridFor(nInc, kThreads), kThreads, 0, s>>>(nInc, w.uStart.p + n, w.uTri.p, w.uIncPtr.p, w.placed.p, w.uInc.p); ++L;
    out.uTri = w.uTri.p; out.uW = w.uW.p; out.incPtr = (int*)w.uIncPtr.p; out.inc = w.uInc.p;
    w.nTouched = 0;
  }
  if (nFloor || w.floorDirty) {
    DCHECK(cudaMemsetAsync(w.floorMult.p, 0, (n + 1) * sizeof(uint32_t), s));
    if (nFloor) { k_floor_mult<<<gridFor(nFloor, kThreads), kThreads, 0, s>>>(nFloor, w.floorList.p, w.floorMult.p); ++L; }
    k_floor_weight<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, w.floorMult.p, w.floorW.p); ++L;
    w.floorDirty = nFloor != 0;
  }
  colliderPass(nFloor != 0);
  DCHECK(dragPass(nFloor || nCol));
  if (nHit || nFloor || nCol || nDrag) {
    DCHECK(w.cDiag.reserve(n + 1));
    const uint32_t nU = nHit;  // bound: the number of distinct contacts is still on its way to the host
    if (nU) {
      DCHECK(w.cPtr.reserve(n + 2)); DCHECK(w.cCol.reserve(6ull * nU + 4)); DCHECK(w.cVal.reserve(6ull * nU + 4));
      k_ccsr_count<<<gridFor(n + 1, kThreads), kThreads, 0, s>>>(n, w.uIncPtr.p, w.uInc.p, w.cPtr.p); ++L;
      L += launchExclusiveScan(s, w.cPtr.p, n + 1, w.scanScratch.p);
    }
    k_ccsr_fill<<<gridFor(n, kThreads), kThreads, 0, s>>>(n, nU ? w.uIncPtr.p : nullptr, w.uInc.p, w.uTri.p, w.uW.p, w.cPtr.p,
                                                         (nFloor || nCol || nDrag) ? w.floorW.p : nullptr, w.cCol.p, w.cVal.p,
                                                         w.cDiag.p); ++L;
    out.cDiag = w.cDiag.p;
    if (nU) { out.cPtr = (int*)w.cPtr.p; out.cCol = w.cCol.p; out.cVal = w.cVal.p; }
  }
  if (nHit) {
    mark(5);
    DCHECK(cudaStreamSynchronize(s));
    mark(6);
    out.nUnique = w.nUnique = (uint32_t)w.host[13];
    if (traceOn)
      std::fprintf(stderr, "[detect] enqueue1 %.0f us, wait1 %.0f | enqueue2 %.0f, wait2 %.0f | enqueue3 %.0f, wait3 %.0f | pairs %llu hits %u\n",
                   stamp[1] - stamp[0], stamp[2] - stamp[1], stamp[3] - stamp[2], stamp[4] - stamp[3], stamp[5] - stamp[4],
                   stamp[6] - stamp[5], (unsigned long long)nPairs, nHit);
  }
  if (launches) *launches += L;
  return 0;
}

// Loads this file's kernels now (CUDA loads a kernel lazily at its first launch; for the collision kernels that
// would be the first contact tick of a run, ~1 ms each in the middle of the simulation).
void preloadDetectKernels() {
  cudaFuncAttributes a;
  cudaFuncGetAttributes(&a, k_tri_ranges);
  cudaFuncGetAttributes(&a, k_floor_write);
  cudaFuncGetAttributes(&a, k_emit_pairs);
  cudaFuncGetAttributes(&a, k_cell_count);
  cudaFuncGetAttributes(&a, k_cell_place);
  cudaFuncGetAttributes(&a, k_cell_rank);
  cudaFuncGetAttributes(&a, k_mark_heads);
  cudaFuncGetAttributes(&a, k_cell_starts);
  cudaFuncGetAttributes(&a, k_pair_filter);
  cudaFuncGetAttributes(&a, k_ccd);
  cudaFuncGetAttributes(&a, k_pair_hits<false>);
  cudaFuncGetAttributes(&a, k_pair_hits<true>);
  cudaFuncGetAttributes(&a, k_inc_count);
  cudaFuncGetAttributes(&a, k_inc_place);
  cudaFuncGetAttributes(&a, k_item_contacts);
  cudaFuncGetAttributes(&a, k_uniq_write);
  cudaFuncGetAttributes(&a, k_item_sort);
  cudaFuncGetAttributes(&a, k_floor_mult);
  cudaFuncGetAttributes(&a, k_floor_weight);
  cudaFuncGetAttributes(&a, k_ccsr_count);
  cudaFuncGetAttributes(&a, k_ccsr_fill);
  cudaFuncGetAttributes(&a, k_init_bbox);
}

}  // namespace pies
