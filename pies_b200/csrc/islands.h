// islands.h — per-substep islands of the global solve and their island-local solves (islands.cu).
#pragma once

#include "engine.h"

namespace pies {

// Island lists of the global solve.  An island is a connected component of S + C_t (static bodies joined by this substep's
// contacts); the system matrix is block diagonal over islands, so every island is an independent solve.  Every island
// goes to one of kIslandLists lists, each solved by its own kind of team (the table in islands.cu), or, when it fits
// none, to the grid-wide CG of pcg.cu.  The list numbers are the slots of pies_b200_debug_island_trace.
constexpr int kIslandLists = 7;

struct IslandWork {
  // once per topology
  DevBuf<uint32_t> bodyOf, rankInBody, bodyPtr, colRank;
  uint32_t nBodies = 0;
  // once per substep
  DevBuf<uint32_t> parent, vals, tmpVals, heads, nodeOff, posOfBody, islStart, order, pos, nnzOff, sortHist, scanScratch;
  DevBuf<uint64_t> keys, tmpKeys;
  DevBuf<uint4> tierDesc;         // per list entry: (island, first row in island order, rows, first matrix entry)
  DevBuf<uint32_t> tierList;      // (kIslandLists + 1) lists of nBodies entries; list kIslandLists = islands left to the global CG
  DevBuf<uint32_t> counts;        // device: [0] islands, [1 + l] islands of list l, [1 + kIslandLists] left over, then nodes
                                  // left over, then inverse floats
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
  uint32_t* host = nullptr;       // pinned copy of counts (11 words)
  uint32_t hostCap = 0;
  cudaEvent_t ready = nullptr;
  // the lists of one solve run beside each other: the first on the solver's stream, the others on these
  static constexpr int kAux = 6;
  cudaStream_t aux[kAux] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t fork = nullptr, join[kAux] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  uint64_t scanCap = 0;
  uint32_t nLeftIslands = 0, nLeftNodes = 0;  // host copies after buildIslands
  uint32_t inverseFloats = 0;                 // floats of inverse (block, dense) one global solve of the island lists reads
  uint32_t listCount[kIslandLists] = {0, 0, 0, 0, 0, 0, 0};
  DevBuf<float> denseInv[kIslandLists];   // dense lists: the inverse of every island's matrix, N x N floats (N: node cap)
  cudaError_t lastError = cudaSuccess;
  ~IslandWork() {
    if (ready) cudaEventDestroy(ready);
    if (fork) cudaEventDestroy(fork);
    for (int k = 0; k < kAux; ++k) { if (join[k]) cudaEventDestroy(join[k]); if (aux[k]) cudaStreamDestroy(aux[k]); }
    if (host) cudaFreeHost(host);
  }
  bool anyLocal() const { for (uint32_t k : listCount) if (k) return true; return false; }   // any island in a list
};

// Upload of the static body tables (HostSystem::bodyOf ...).
int uploadIslandStatics(IslandWork& w, cudaStream_t s, const HostSystem& y);

// Builds this substep's islands from the contact lists and sorts them into the lists.  Synchronises the stream once (the
// host needs to know whether any island is left to the global CG).  slotOf / blockCount: this substep's preconditioner
// blocks (reblock.cu).  tuning: PiesB200Tuning::reserved, whose island bits choose the lists in use.  Returns 0 or -1.
int buildIslands(IslandWork& w, cudaStream_t s, uint32_t n, const CsrMatrix& S, const ContactLists& c,
                 const uint32_t* slotOf, const uint32_t* blockCount, uint32_t nBlocksBound, uint32_t tuning, int* launches);

// The island counts of the last buildIslands in the public statistics (islandsTier, islandsGlobal, ...).
void islandStats(const IslandWork& w, PiesB200Stats& st);

// Solves A x = b on every island of the lists (x holds the start value).  statSlot: which 4-word record of solveStats.
int launchIslandSolve(IslandWork& w, cudaStream_t s, const CsrMatrix& S, const ContactLists& c, const PcgWork& pw,
                      const uint32_t* slotOf, const float4* b, float4* x, float tol, uint32_t maxIter, uint32_t statSlot);

// Points pw at the active-row tables when this substep's grid-wide solve is restricted to the left-over islands.
void applyRestriction(const IslandWork& w, PcgWork& pw);

void preloadIslandKernels();

}  // namespace pies
