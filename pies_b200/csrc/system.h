// system.h — once-per-topology host precomputation for the PD global/local steps.
#pragma once

#include <cstdint>
#include <vector>

#include "kernels.h"
#include "scene.h"

namespace pies {

struct HostSystem {
  uint32_t n = 0;

  // fused tet elements (strain + volume on the same tet share one record), plane layout of kernels.h
  uint32_t nElems = 0;
  std::vector<uint32_t> elemIds;              // 4 per element
  std::vector<float> elemQa, elemQb, elemPc, elemPd;  // 4 floats per element each

  // contribution slots (one float4 each) and the per-node gather lists
  uint64_t baseTet = 0, baseDist = 0, baseBend = 0, baseShape = 0, baseGoal = 0, basePos = 0, nContrib = 0;
  std::vector<float> posContrib;              // constant w * fixedPosition, 4 floats per position constraint
  std::vector<int> incPtr;                    // n + 1
  std::vector<uint32_t> inc;

  // S = M/h^2 + sum w A^T A  (reference Solver.cpp:174-210), CSR with both triangles
  std::vector<int> rowPtr, col;
  std::vector<float> val;

  // The same matrix for the CG mat-vec, sliced ELLPACK (SELL-32-sigma): rows are sorted by length inside windows of
  // kSellWindow consecutive rows, cut into slices of 32 (one warp), every slice padded to its longest row and stored
  // column-major, so lane l reads entry k of its row at sellPtr[s] + 32 k + l: coalesced, no staging, no divergence.
  // Entries of a row keep their CSR order.
  std::vector<uint32_t> sellPtr;              // nSlices + 1 element offsets (multiples of 32)
  std::vector<uint32_t> sellRow;              // 32 per slice, 0xffffffff = padding lane
  std::vector<int> sellCol;                   // padded entries: column = the row itself, value = 0
  std::vector<float> sellVal;
  static constexpr uint32_t kSellWindow = 256;   // == rows one CTA of k_pcg_spmv stages per step (pcg.cu kWinRows)

  // block-Jacobi preconditioner
  uint32_t nBlocks = 0;
  std::vector<int> blockNodes;                // 32 per block, -1 padded
  std::vector<float> blockInv;                // 1024 per block, symmetric

  // Static bodies: connected components of S (nodes that also share a preconditioner block are kept together).
  // The per-substep islands of the global solve (islands.cu) are unions of bodies joined by contacts.  Bodies are
  // numbered by their smallest node; bodyNodes lists every body's nodes in ascending order.
  uint32_t nBodies = 0;
  std::vector<uint32_t> bodyOf;               // n: node -> body
  std::vector<uint32_t> rankInBody;           // n: node -> position inside bodyNodes[bodyPtr[b] ..)
  std::vector<uint32_t> bodyPtr;              // nBodies + 1
  std::vector<uint32_t> bodyNodes;            // n
  // per CSR entry of S: rankInBody of its column (S never leaves a body), 0xffffffff for an explicit zero that points
  // outside the row's body (bend stencils); lets the island solver re-index a row without a gather per entry
  std::vector<uint32_t> colRank;

  // Closed segments of the fused local step + RHS (k_tet_rhs, one CTA per segment).  A segment is a run of whole bodies
  // whose nodes are one index range [n0, n1) and whose fused tet elements are one range [e0, e1), such that the elements
  // reference only nodes of [n0, n1) and every incidence of those nodes is a tet slot of an element in [e0, e1) (no
  // other constraint type touches them), and at most kSegElems elements and kSegNodes nodes (kernels.h).  Its
  // contributions then never have to leave the CTA.  Bodies that break a condition keep the two-kernel path: their
  // elements are listed in restElems, their nodes in restNodes (both ascending).
  std::vector<uint32_t> segs;                 // 4 per segment: n0, n1, e0, e1
  std::vector<uint16_t> segSlot;              // parallel to inc: 4 (e - e0) + k for an incidence of a segment node, else 0
  std::vector<uint32_t> restElems, restNodes;

  uint64_t staticProjections = 0;             // per PD iteration, shape/goal count one per member
};

// Fills the segment fields of a HostSystem whose elements and gather lists are built.  O(n + incidences).
void buildSegments(HostSystem& y);

// Sliced-ELLPACK copy of a CSR matrix (layout described in HostSystem).  Host only.
void buildSell(uint32_t n, const int* rowPtr, const int* col, const float* val, std::vector<uint32_t>& sellPtr,
               std::vector<uint32_t>& sellRow, std::vector<int>& sellCol, std::vector<float>& sellVal);

// h = fixedTimestepSize / timeSubsteps.  threads: worker threads for the row-wise assembly.
void buildSystem(const HostScene& sc, float h, HostSystem& out, unsigned threads);

}  // namespace pies
