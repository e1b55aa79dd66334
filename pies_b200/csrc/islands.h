// islands.h — per-substep islands of the global solve and their island-local solves (islands.cu).
#pragma once

#include "engine.h"

namespace pies {

// Tiers of the island-local solve.  An island is a connected component of S + C_t (static bodies joined by this
// substep's contacts); the system matrix is block diagonal over islands, so every island is an independent solve.
//   tier 0: one warp per island (<= 32 nodes in a single preconditioner block: every free body of the S3 stack),
//           iterative refinement with the block's exact inverse
//   tier 1: one 320-thread CTA running CG, matrix + block inverses + r, p resident in shared memory, two CTAs per SM
//   tier 2: one 512-thread CTA, the same with the whole shared memory of an SM
//   tier 3: one 1024-thread CTA, r and p in shared memory, the island's matrix re-indexed in a global scratch copy
//           (L2 resident: one CTA re-reads a few hundred KB per iteration)
// Islands above tier 3 are left to the grid-wide CG of pcg.cu.
// Tier 1 has a second, internal list (slot 4): islands of at most 256 nodes go to a 128-thread CTA with the same
// shared-memory layout, five CTAs per SM — at S3 the typical contact island is five bodies (~140 rows), which leaves more
// than half of a 320-thread CTA waiting at every barrier.  The public statistics and tuning bits count it as tier 1.
// A third internal list (slot 5) takes the islands of at most 128 nodes that are not a single preconditioner block: their
// matrix is inverted once per substep (dense, in-place Gauss-Jordan, one CTA per island) and every global solve of the
// substep is then iterative refinement with that inverse — what the warp tier does with its block inverse.  At S3 every
// contact island of the benchmark window (3-4 bodies of a column, 81-108 nodes) is of this kind.
constexpr int kIslandTiers = 4;
// A second dense list (slot 6) does the same for islands of 129..192 nodes with a 576-thread inversion CTA (a column of
// 5-7 bodies: S3 ticks 79..100); beyond that the m^3 of the inversion and the m^2 of every apply lose to the CG.
constexpr int kIslandSlots = kIslandTiers + 3;
constexpr int kSmallCtaSlot = 4;
constexpr int kDenseSlot = 5;         // <= kDenseMax nodes
constexpr int kDenseSlot2 = 6;        // <= kDenseMax2 nodes
constexpr uint32_t kDenseMax = 128;   // nodes; the inverse is stored with this leading dimension
constexpr uint32_t kDenseMax2 = 192;
struct IslandCaps { uint32_t maxNodes, maxNnz, maxInv, maxBlocks; };

struct IslandWork {
  // once per topology
  DevBuf<uint32_t> bodyOf, rankInBody, bodyPtr, colRank;
  uint32_t nBodies = 0;
  // once per substep
  DevBuf<uint32_t> parent, vals, tmpVals, heads, nodeOff, posOfBody, islStart, order, pos, nnzOff, sortHist, scanScratch;
  DevBuf<uint64_t> keys, tmpKeys;
  DevBuf<uint4> tierDesc;         // per list entry: (island, first row in island order, rows, first matrix entry)
  DevBuf<uint32_t> tierList;      // (kIslandSlots + 1) lists of nBodies entries; list kIslandSlots = islands left to the global CG
  DevBuf<uint32_t> counts;        // device: [0] islands, [1 + t] islands of list t, [1 + kIslandSlots] left over, then nodes left over
  DevBuf<uint32_t> blkLocal;      // preconditioner block * 32 + lane -> island-local row of that member (written by every solve)
  DevBuf<uint32_t> slotIsl;       // tier 3: preconditioner slot of every row, island order
  DevBuf<int> matCol;             // tier 3: island-local copy of the matrix (column = local row index), at nnzOff
  DevBuf<float> matVal;
  // restriction of the grid-wide CG to the islands left over (PcgWork::big / actWin / actBlk): built when both kinds exist
  DevBuf<uint8_t> big;
  DevBuf<uint32_t> winFlag, blkFlag, actWin, actBlk, actCounts;
  bool restricted = false;
  bool united = false;            // this substep's islands were built from contacts (parent holds the forest over bodies)
  DevBuf<uint4> trace;            // diagnostics (PIES_B200_ISLAND_TRACE): per list entry (rows, iterations, SM clocks, matrix entries) of the last solve
  DevBuf<uint32_t> solveStats;    // 4 words per solve of a tick: max iterations, sum of iterations x rows, islands at the cap, worst residual
  uint32_t* host = nullptr;       // pinned copy of counts (8 words) + solveStats
  uint32_t hostCap = 0;
  cudaEvent_t ready = nullptr;
  // the lists of one solve run beside each other: the first on the solver's stream, the others on these
  static constexpr int kAux = 6;
  cudaStream_t aux[kAux] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[kAux] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  uint64_t scanCap = 0;
  uint32_t nLeftIslands = 0, nLeftNodes = 0;  // host copies after buildIslands
  uint32_t inverseFloats = 0;                 // floats of inverse (block, dense) one global solve of the island lists reads
  uint32_t tierCount[kIslandSlots] = {0, 0, 0, 0, 0, 0, 0};
  DevBuf<float> denseInv, denseInv2;   // slots 5 / 6: N x N floats per list entry (N = kDenseMax / kDenseMax2), inverse of the island's matrix
  cudaError_t lastError = cudaSuccess;
  ~IslandWork() {
    if (ready) cudaEventDestroy(ready);
    if (fork) cudaEventDestroy(fork);
    for (int k = 0; k < kAux; ++k) { if (join[k]) cudaEventDestroy(join[k]); if (aux[k]) cudaStreamDestroy(aux[k]); }
    if (host) cudaFreeHost(host);
  }
};

// Upload of the static body tables (HostSystem::bodyOf ...).
int uploadIslandStatics(IslandWork& w, cudaStream_t s, const HostSystem& y);

// Builds this substep's islands from the contact lists and classifies them.  Synchronises the stream once (the host
// needs to know whether any island is left to the global CG).  slotOf / blockCount: this substep's preconditioner
// blocks (reblock.cu).  Returns 0 or -1.
int buildIslands(IslandWork& w, cudaStream_t s, uint32_t n, const CsrMatrix& S, const ContactLists& c,
                 const uint32_t* slotOf, const uint32_t* blockCount, uint32_t nBlocksBound, uint32_t tiersEnabled,
                 int* launches);

// Solves A x = b on every island of tiers 0..3 (x holds the start value).  statSlot: which 4-word record of solveStats.
int launchIslandSolve(IslandWork& w, cudaStream_t s, const CsrMatrix& S, const ContactLists& c, const PcgWork& pw,
                      const uint32_t* slotOf, const float4* b, float4* x, float tol, uint32_t maxIter, uint32_t statSlot);

// Points pw at the active-row tables when this substep's grid-wide solve is restricted to the left-over islands.
void applyRestriction(const IslandWork& w, PcgWork& pw);

void preloadIslandKernels();

}  // namespace pies
