// detect.h — work buffers and entry point of the once-per-substep collision detection.
#pragma once

#include <algorithm>

#include "engine.h"

namespace pies {

struct DetectInput {
  const uint32_t* tri;   // 3 node ids per triangle (device)
  const float4* q;       // current positions
  const float4* prev;    // positions at the start of the substep
  uint32_t nTri, nNodes, threadCount;
  float threshold;       // collisionThresholdDistance
  float floorLimit;      // floorHeight + collisionThickness
  const uint32_t* order = nullptr;  // optional canonical-order override (device), see canonicalRank
  ColliderSet colliders{};          // static colliders (colliders.cu): masks into colMask, weights into floorW
  float thickness = 0.0f;           // collisionThickness
  uint32_t* colMask = nullptr;
  DragSet drags{};                  // drag targets (pick.cu): weights into floorW after the colliders', w g into msn
  float4* msn = nullptr;
};

struct DetectWork {
  DevBuf<int4> triMin;
  DevBuf<uint4> triRec;                         // (a, b, c, lx | ly << 8 | lz << 16)
  DevBuf<uint32_t> cnt, cntRank, floorRank, hitCount, scanScratch;
  DevBuf<float4> aabbLo, aabbHi;
  DevBuf<int> bbox;
  DevBuf<uint64_t> keys, tmpKeys;
  DevBuf<uint32_t> vals /* sorted: member triangle of every (cell, member) pair */, tmpVals, heads, cellStart, sortHist,
      ticket, nodeDone;
  // node incidence (counting sort): arrival numbers, placed items, per-item scratch of the distinct-contact ranking
  DevBuf<uint32_t> arrival, placed, pointTri, headTri, uMult;
  // small grids: direct cell table (counts -> starts), arrival numbers and unordered placement of the (cell, triangle) pairs
  DevBuf<uint32_t> cellTable, arrivalP, placedP;
  DevBuf<uint4> triList, uTri;     // full list (canonical order) and distinct contacts
  DevBuf<uint32_t> otherTri, uStart, uIncPtr, uInc, pairSlot;
  DevBuf<uint8_t> candHit;
  DevBuf<uint2> cand, pairRun;      // candidate (point node, triangle) pairs of the narrow phase (cell-sorted chunks) and every pair's run
  uint32_t candCap = 0;
  DevBuf<float> uW;
  uint32_t nUnique = 0, nTouched = 0;
  DevBuf<uint32_t> floorList, incPtr, floorMult;
  DevBuf<float> floorW;
  // contact matrix C_t of the substep as CSR (off-diagonals) + per-node diagonal (contacts + floor), see k_ccsr_fill
  DevBuf<uint32_t> cPtr; DevBuf<int> cCol; DevBuf<float> cVal, cDiag;
  int* host = nullptr;   // pinned, 16 ints
  uint64_t nPairs = 0, scanCap = 0;
  uint32_t nCells = 0;
  int keyPack[5] = {0, 0, 0, 0, 0};  // minX, minY, minZ, bitsY, bitsZ of the last detection
  bool failed = false, badInput = false, floorDirty = true;
  cudaError_t lastError = cudaSuccess;
};

// Fills `out` (device pointers owned by `w`) with the point-triangle and floor lists in the
// reference's canonical order plus the node->entry incidence table.  Returns 0, or -1 on a CUDA error.
int detectTriangles(DetectWork& w, cudaStream_t s, const DetectInput& in, ContactLists& out, int* launches);

}  // namespace pies
