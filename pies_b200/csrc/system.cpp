// system.cpp — once-per-topology host precomputation.
//
// Mirrors what the reference does when the node count changes (reference
// Src/Solver.cpp:168-221): it assembles S = M/h^2 + sum_i w_i A_i^T A_i with the same
// per-coefficient accumulation order as the reference's coeffRef(i,j) += sequence
// (mass diagonal, position, distance, tet, volume, shape, goal, bend; Solver.cpp:179-210),
// but in O(nnz) instead of the reference's quadratic sparse insertion (SURVEY F15).
// In place of the Cholesky factor it prepares a block-Jacobi preconditioner, and for the
// local step it fuses strain/volume constraints that sit on the same tet and builds the
// vertex -> contribution gather lists (deterministic RHS assembly).
#include "system.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include <thread>
#include <unordered_map>

namespace pies {
namespace {

struct TetKey {
  uint32_t w[13];
  bool operator==(const TetKey& o) const { return std::memcmp(w, o.w, sizeof(w)) == 0; }
};
struct TetKeyHash {
  size_t operator()(const TetKey& k) const {
    uint64_t h = 1469598103934665603ull;
    for (uint32_t v : k.w) { h ^= v; h *= 1099511628211ull; }
    return (size_t)h;
  }
};
TetKey makeKey(const uint32_t* ids, const float* qinv) {
  TetKey k;
  std::memcpy(k.w, ids, 16);
  std::memcpy(k.w + 4, qinv, 36);
  return k;
}

// w * A^T A of a tet-type constraint (Constraints.cpp:141-175, Constraints.h:58): A has a zero first
// row and rows 1..3 = Qinv^T [-1 | I].
void tetAtA(const float* qinv, float out[4][4]) {
  float A[3][4];
  for (int r = 0; r < 3; ++r) {
    float d0 = qinv[3 * r], d1 = qinv[3 * r + 1], d2 = qinv[3 * r + 2];
    A[r][0] = ((-d0) + (-d1)) + (-d2);
    A[r][1] = d0; A[r][2] = d1; A[r][3] = d2;
  }
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) out[i][j] = A[0][i] * A[0][j] + A[1][i] * A[1][j] + A[2][i] * A[2][j];
}

struct Dsu {
  std::vector<uint32_t> p;
  explicit Dsu(uint32_t n) : p(n) { std::iota(p.begin(), p.end(), 0u); }
  uint32_t find(uint32_t x) { while (p[x] != x) { p[x] = p[p[x]]; x = p[x]; } return x; }
  void unite(uint32_t a, uint32_t b) { a = find(a); b = find(b); if (a != b) p[std::max(a, b)] = std::min(a, b); }
};

}  // namespace

// Sliced ELLPACK (SELL-32-sigma) copy of a CSR matrix, see system.h.
void buildSell(uint32_t n, const int* rowPtr, const int* col, const float* val, std::vector<uint32_t>& sellPtr,
               std::vector<uint32_t>& sellRow, std::vector<int>& sellCol, std::vector<float>& sellVal) {
  const uint32_t nSlices = (n + 31u) / 32u;
  std::vector<uint32_t> order(n);
  for (uint32_t i = 0; i < n; ++i) order[i] = i;
  auto len = [&](uint32_t r) { return (uint32_t)(rowPtr[r + 1] - rowPtr[r]); };
  for (uint32_t w0 = 0; w0 < n; w0 += HostSystem::kSellWindow) {
    uint32_t w1 = std::min(n, w0 + HostSystem::kSellWindow);
    std::stable_sort(order.begin() + w0, order.begin() + w1, [&](uint32_t a, uint32_t b) { return len(a) > len(b); });
  }
  sellPtr.assign(nSlices + 1, 0);
  sellRow.assign((size_t)nSlices * 32, 0xffffffffu);
  for (uint32_t sl = 0; sl < nSlices; ++sl) {
    uint32_t longest = 0;
    for (uint32_t l = 0; l < 32 && sl * 32 + l < n; ++l) {
      sellRow[(size_t)sl * 32 + l] = order[sl * 32 + l];
      longest = std::max(longest, len(order[sl * 32 + l]));
    }
    sellPtr[sl + 1] = sellPtr[sl] + 32u * longest;
  }
  sellCol.assign(sellPtr[nSlices], 0);
  sellVal.assign(sellPtr[nSlices], 0.0f);
  for (uint32_t sl = 0; sl < nSlices; ++sl) {
    const uint32_t longest = (sellPtr[sl + 1] - sellPtr[sl]) / 32u;
    for (uint32_t l = 0; l < 32; ++l) {
      const uint32_t r = sellRow[(size_t)sl * 32 + l];
      const uint32_t m = r == 0xffffffffu ? 0u : len(r);
      for (uint32_t k = 0; k < longest; ++k) {
        const size_t idx = (size_t)sellPtr[sl] + 32u * k + l;
        if (k < m) { sellCol[idx] = col[rowPtr[r] + k]; sellVal[idx] = val[rowPtr[r] + k]; }
        else sellCol[idx] = r == 0xffffffffu ? 0 : (int)r;
      }
    }
  }
}

void buildSegments(HostSystem& y) {
  y.segs.clear(); y.restElems.clear(); y.restNodes.clear();
  y.segSlot.assign(y.inc.size(), 0);
  const uint64_t tetEnd = y.baseTet + 4ull * y.nElems;
  constexpr uint32_t kNone = 0xffffffffu;
  uint32_t cur[4] = {0, 0, kNone, kNone};  // open segment: n0, n1, e0, e1 (e0 == kNone: no element yet)
  bool open = false;
  auto close = [&]() {
    if (!open) return;
    if (cur[2] == kNone) cur[2] = cur[3] = 0;
    y.segs.insert(y.segs.end(), cur, cur + 4);
    open = false;
  };
  for (uint32_t b = 0; b < y.nBodies; ++b) {
    const uint32_t p0 = y.bodyPtr[b], cnt = y.bodyPtr[b + 1] - p0, a = y.bodyNodes[p0];
    bool ok = y.bodyNodes[p0 + cnt - 1] - a + 1 == cnt && cnt <= kSegNodes;  // bodyNodes is ascending
    uint32_t eLo = kNone, eHi = 0;
    for (uint32_t i = a; ok && i < a + cnt; ++i)
      for (int k = y.incPtr[i]; k < y.incPtr[i + 1]; ++k) {
        const uint64_t slot = y.inc[k];
        if (slot < y.baseTet || slot >= tetEnd) { ok = false; break; }
        const uint32_t e = (uint32_t)((slot - y.baseTet) / 4);
        eLo = std::min(eLo, e); eHi = std::max(eHi, e);
      }
    const bool hasElems = eLo != kNone;
    ok = ok && (!hasElems || eHi - eLo + 1 <= kSegElems);
    for (uint32_t e = eLo; ok && hasElems && e <= eHi; ++e)   // the range holds no element of another body
      for (int k = 0; k < 4; ++k) {
        const uint32_t v = y.elemIds[4ull * e + k];
        if (v < a || v >= a + cnt) { ok = false; break; }
      }
    if (!ok) { close(); continue; }
    const uint32_t nE = hasElems ? eHi + 1 - eLo : 0;
    const uint32_t curE = cur[2] == kNone ? 0 : cur[3] - cur[2];
    const bool joins = open && a == cur[1] && cur[1] - cur[0] + cnt <= kSegNodes &&
                       curE + nE <= kSegElems && (!hasElems || cur[2] == kNone || eLo == cur[3]);
    if (!joins) {
      close();
      cur[0] = cur[1] = a; cur[2] = cur[3] = kNone;
      open = true;
    }
    cur[1] = a + cnt;
    if (hasElems) {
      if (cur[2] == kNone) cur[2] = eLo;
      cur[3] = eHi + 1;
    }
  }
  close();
  std::vector<char> nodeIn(y.n, 0), elemIn(y.nElems, 0);
  for (size_t s = 0; s < y.segs.size(); s += 4) {
    const uint32_t n0 = y.segs[s], n1 = y.segs[s + 1], e0 = y.segs[s + 2], e1 = y.segs[s + 3];
    for (uint32_t i = n0; i < n1; ++i) {
      nodeIn[i] = 1;
      for (int k = y.incPtr[i]; k < y.incPtr[i + 1]; ++k) y.segSlot[k] = (uint16_t)(y.inc[k] - y.baseTet - 4ull * e0);
    }
    for (uint32_t e = e0; e < e1; ++e) elemIn[e] = 1;
  }
  for (uint32_t i = 0; i < y.n; ++i) if (!nodeIn[i]) y.restNodes.push_back(i);
  for (uint32_t e = 0; e < y.nElems; ++e) if (!elemIn[e]) y.restElems.push_back(e);
}

void buildSystem(const HostScene& sc, float h, HostSystem& out, unsigned threads) {
  out = HostSystem{};
  const uint32_t n = sc.nodeCount();
  out.n = n;
  const float h2 = h * h;
  const size_t nPos = sc.posW.size(), nDist = sc.distW.size(), nTet = sc.tetW.size(), nVol = sc.volW.size(),
               nBend = sc.bendW.size(), nShapeM = sc.shapeId.size(), nGoalM = sc.goalId.size();

  // ---- 1. fuse strain + volume constraints sitting on the same tet ------------------------------
  std::vector<int64_t> volOfTet(nTet, -1);
  std::vector<char> volUsed(nVol, 0);
  {
    bool aligned = nTet == nVol;
    for (size_t i = 0; aligned && i < nTet; ++i)
      aligned = std::memcmp(&sc.tetId[4 * i], &sc.volId[4 * i], 16) == 0 &&
                std::memcmp(&sc.tetQinv[9 * i], &sc.volQinv[9 * i], 36) == 0;
    if (aligned) {
      for (size_t i = 0; i < nTet; ++i) { volOfTet[i] = (int64_t)i; volUsed[i] = 1; }
    } else {
      std::unordered_multimap<TetKey, uint32_t, TetKeyHash> map;
      map.reserve(nVol * 2);
      for (size_t j = nVol; j-- > 0;) map.emplace(makeKey(&sc.volId[4 * j], &sc.volQinv[9 * j]), (uint32_t)j);
      for (size_t i = 0; i < nTet; ++i) {
        auto it = map.find(makeKey(&sc.tetId[4 * i], &sc.tetQinv[9 * i]));
        if (it != map.end()) { volOfTet[i] = it->second; volUsed[it->second] = 1; map.erase(it); }
      }
    }
  }
  auto pushElem = [&](const uint32_t* ids, const float* qi, float wS, float lo, float hi, float wV, float oLo, float oHi) {
    out.elemIds.insert(out.elemIds.end(), ids, ids + 4);
    out.elemQa.insert(out.elemQa.end(), qi, qi + 4);
    out.elemQb.insert(out.elemQb.end(), qi + 4, qi + 8);
    const float pc[4] = {qi[8], wS, lo, hi}, pd[4] = {wV, oLo, oHi, 0.0f};
    out.elemPc.insert(out.elemPc.end(), pc, pc + 4);
    out.elemPd.insert(out.elemPd.end(), pd, pd + 4);
  };
  out.elemIds.reserve(4 * (nTet + nVol));
  for (size_t i = 0; i < nTet; ++i) {
    int64_t v = volOfTet[i];
    pushElem(&sc.tetId[4 * i], &sc.tetQinv[9 * i], sc.tetW[i], sc.tetMin[i], sc.tetMax[i], v >= 0 ? sc.volW[v] : 0.0f,
             v >= 0 ? sc.volMin[v] : 1.0f, v >= 0 ? sc.volMax[v] : 1.0f);
  }
  for (size_t j = 0; j < nVol; ++j)
    if (!volUsed[j]) pushElem(&sc.volId[4 * j], &sc.volQinv[9 * j], 0.0f, 0.0f, 0.0f, sc.volW[j], sc.volMin[j], sc.volMax[j]);
  out.nElems = (uint32_t)(out.elemIds.size() / 4);

  // ---- 2. contribution slots + gather lists (reference RHS order: Solver.cpp:310-335) -----------------
  out.baseTet = 0;
  out.baseDist = out.baseTet + 4ull * out.nElems;
  out.baseBend = out.baseDist + 2ull * nDist;
  out.baseShape = out.baseBend + 4ull * nBend;
  out.baseGoal = out.baseShape + nShapeM;
  out.basePos = out.baseGoal + nGoalM;
  out.nContrib = out.basePos + nPos;
  out.posContrib.resize(4 * nPos);
  for (size_t c = 0; c < nPos; ++c) {
    for (int k = 0; k < 3; ++k) out.posContrib[4 * c + k] = sc.posW[c] * sc.posTarget[3 * c + k];
    out.posContrib[4 * c + 3] = 0.0f;
  }
  out.incPtr.assign(n + 1, 0);
  auto forEachIncidence = [&](auto&& fn) {  // fn(node, slot) in the reference's RHS summation order
    for (size_t c = 0; c < nPos; ++c) fn(sc.posId[c], out.basePos + c);
    for (size_t c = 0; c < nDist; ++c) for (int k = 0; k < 2; ++k) fn(sc.distId[2 * c + k], out.baseDist + 2 * c + k);
    for (size_t e = 0; e < out.nElems; ++e) for (int k = 0; k < 4; ++k) fn(out.elemIds[4 * e + k], out.baseTet + 4 * e + k);
    for (size_t c = 0; c < nBend; ++c) for (int k = 0; k < 4; ++k) fn(sc.bendId[4 * c + k], out.baseBend + 4 * c + k);
    for (size_t m = 0; m < nShapeM; ++m) fn(sc.shapeId[m], out.baseShape + m);
    for (size_t m = 0; m < nGoalM; ++m) fn(sc.goalId[m], out.baseGoal + m);
  };
  forEachIncidence([&](uint32_t node, uint64_t) { ++out.incPtr[node + 1]; });
  for (uint32_t i = 0; i < n; ++i) out.incPtr[i + 1] += out.incPtr[i];
  out.inc.resize(out.incPtr[n]);
  {
    std::vector<int> cur(out.incPtr.begin(), out.incPtr.end() - 1);
    forEachIncidence([&](uint32_t node, uint64_t slot) { out.inc[cur[node]++] = (uint32_t)slot; });
  }
  out.staticProjections = nPos + nDist + nTet + nVol + nBend + nShapeM + nGoalM;

  // ---- 3. S in CSR, coefficient sums in the reference's accumulation order ---------------------------
  std::vector<uint32_t> rowCount(n + 1, 0);
  auto forEachCoeff = [&](auto&& fn) {  // fn(row, col, value)
    for (uint32_t i = 0; i < n; ++i) fn(i, i, 1.0f / (sc.invMass[i] * h2));
    for (size_t c = 0; c < nPos; ++c) fn(sc.posId[c], sc.posId[c], sc.posW[c] * 1.0f);
    for (size_t c = 0; c < nDist; ++c) {
      const float AtA[2][2] = {{0.5f, -0.5f}, {-0.5f, 0.5f}};
      for (int i = 0; i < 2; ++i) for (int j = 0; j < 2; ++j) fn(sc.distId[2 * c + i], sc.distId[2 * c + j], sc.distW[c] * AtA[i][j]);
    }
    float M[4][4];
    for (size_t c = 0; c < nTet; ++c) {
      tetAtA(&sc.tetQinv[9 * c], M);
      for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) fn(sc.tetId[4 * c + i], sc.tetId[4 * c + j], sc.tetW[c] * M[i][j]);
    }
    for (size_t c = 0; c < nVol; ++c) {
      tetAtA(&sc.volQinv[9 * c], M);
      for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) fn(sc.volId[4 * c + i], sc.volId[4 * c + j], sc.volW[c] * M[i][j]);
    }
    for (size_t k = 0; k + 1 < sc.shapeOff.size(); ++k)
      for (uint32_t m = sc.shapeOff[k]; m < sc.shapeOff[k + 1]; ++m) fn(sc.shapeId[m], sc.shapeId[m], sc.shapeW[k]);
    for (size_t k = 0; k + 1 < sc.goalOff.size(); ++k)
      for (uint32_t m = sc.goalOff[k]; m < sc.goalOff[k + 1]; ++m) fn(sc.goalId[m], sc.goalId[m], sc.goalW[k]);
    for (size_t c = 0; c < nBend; ++c)
      for (int i = 0; i < 4; ++i) for (int j = 0; j < 4; ++j) fn(sc.bendId[4 * c + i], sc.bendId[4 * c + j], sc.bendW[c] * (i == j ? 1.0f : 0.0f));
  };
  forEachCoeff([&](uint32_t r, uint32_t, float) { ++rowCount[r + 1]; });
  std::vector<uint64_t> rowStart(n + 1, 0);
  for (uint32_t i = 0; i < n; ++i) rowStart[i + 1] = rowStart[i] + rowCount[i + 1];
  std::vector<uint32_t> rawCol(rowStart[n]);
  std::vector<float> rawVal(rowStart[n]);
  {
    std::vector<uint64_t> cur(rowStart.begin(), rowStart.end() - 1);
    forEachCoeff([&](uint32_t r, uint32_t c, float v) { uint64_t k = cur[r]++; rawCol[k] = c; rawVal[k] = v; });
  }
  // per row: stable order by column, then sum duplicates front to back (== coeffRef += order)
  std::vector<uint32_t> uniq(n, 0);
  unsigned T = std::max(1u, threads);
  auto compactRows = [&](unsigned t) {
    std::vector<uint32_t> order;
    std::vector<uint32_t> tc;
    std::vector<float> tv;
    for (uint32_t r = t; r < n; r += T) {
      uint64_t b = rowStart[r], e = rowStart[r + 1];
      size_t m = e - b;
      order.resize(m);
      std::iota(order.begin(), order.end(), 0u);
      std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return rawCol[b + x] < rawCol[b + y]; });
      tc.clear(); tv.clear();
      for (size_t k = 0; k < m; ++k) {
        uint32_t c = rawCol[b + order[k]];
        float v = rawVal[b + order[k]];
        if (!tc.empty() && tc.back() == c) tv.back() += v; else { tc.push_back(c); tv.push_back(v); }
      }
      // bend constraints add explicit zeros off the diagonal in the reference too; keep them (harmless)
      for (size_t k = 0; k < tc.size(); ++k) { rawCol[b + k] = tc[k]; rawVal[b + k] = tv[k]; }
      uniq[r] = (uint32_t)tc.size();
    }
  };
  {
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < T; ++t) pool.emplace_back(compactRows, t);
    compactRows(0);
    for (auto& th : pool) th.join();
  }
  out.rowPtr.assign(n + 1, 0);
  for (uint32_t i = 0; i < n; ++i) out.rowPtr[i + 1] = out.rowPtr[i] + (int)uniq[i];
  out.col.resize(out.rowPtr[n]);
  out.val.resize(out.rowPtr[n]);
  for (uint32_t r = 0; r < n; ++r)
    for (uint32_t k = 0; k < uniq[r]; ++k) {
      out.col[out.rowPtr[r] + k] = (int)rawCol[rowStart[r] + k];
      out.val[out.rowPtr[r] + k] = rawVal[rowStart[r] + k];
    }
  rawCol.clear(); rawCol.shrink_to_fit();
  rawVal.clear(); rawVal.shrink_to_fit();

  // ---- 3b. sliced ELLPACK copy for the CG mat-vec -----------------------------------------------------
  buildSell(n, out.rowPtr.data(), out.col.data(), out.val.data(), out.sellPtr, out.sellRow, out.sellCol, out.sellVal);

  // ---- 4. block-Jacobi preconditioner: blocks of <= 32 nodes following connectivity ------------------
  Dsu dsu(n);
  for (uint32_t r = 0; r < n; ++r)
    for (int k = out.rowPtr[r]; k < out.rowPtr[r + 1]; ++k)
      if (out.val[k] != 0.0f) dsu.unite(r, (uint32_t)out.col[k]);
  // component member lists in ascending node order
  std::vector<uint32_t> root(n), compSize(n, 0);
  for (uint32_t i = 0; i < n; ++i) { root[i] = dsu.find(i); ++compSize[root[i]]; }
  std::vector<int> blockOf(n, -1);
  std::vector<int>& bn = out.blockNodes;
  auto newBlock = [&]() { bn.insert(bn.end(), 32, -1); return (int)(bn.size() / 32 - 1); };
  int openBlock = -1, openFill = 0;  // small components are packed together
  std::vector<char> visited(n, 0);
  std::vector<uint32_t> queue;
  for (uint32_t i = 0; i < n; ++i) {
    if (visited[i]) continue;
    uint32_t sz = compSize[root[i]];
    // breadth-first order through S so that consecutive chunks of a large body are compact
    queue.clear();
    queue.push_back(i);
    visited[i] = 1;
    for (size_t head = 0; head < queue.size(); ++head) {
      uint32_t u = queue[head];
      for (int k = out.rowPtr[u]; k < out.rowPtr[u + 1]; ++k) {
        uint32_t v = (uint32_t)out.col[k];
        if (!visited[v] && out.val[k] != 0.0f) { visited[v] = 1; queue.push_back(v); }
      }
    }
    if (sz <= 32) {
      if (openBlock < 0 || openFill + (int)sz > 32) { openBlock = newBlock(); openFill = 0; }
      for (uint32_t u : queue) { bn[32 * openBlock + openFill] = (int)u; blockOf[u] = openBlock; ++openFill; }
      if (sz > 16) openBlock = -1;  // do not bother topping up mostly-full blocks
    } else {
      for (size_t k = 0; k < queue.size(); k += 32) {
        int b = newBlock();
        for (size_t j = k; j < std::min(queue.size(), k + 32); ++j) { bn[32 * b + (j - k)] = (int)queue[j]; blockOf[queue[j]] = b; }
      }
    }
  }
  out.nBlocks = (uint32_t)(bn.size() / 32);
  // ---- 4b. static bodies (the units the per-substep islands are made of) -----------------------------------
  {
    for (uint32_t b = 0; b < out.nBlocks; ++b)  // small components packed into one block stay together
      for (int k = 1; k < 32 && bn[32 * b + k] >= 0; ++k) dsu.unite((uint32_t)bn[32 * b], (uint32_t)bn[32 * b + k]);
    out.bodyOf.assign(n, 0);
    out.rankInBody.assign(n, 0);
    std::vector<uint32_t> bodyOfRoot(n, 0xffffffffu);
    out.nBodies = 0;
    for (uint32_t i = 0; i < n; ++i) {  // min-hooking: a root is its body's smallest node, so bodies come out in node order
      const uint32_t r = dsu.find(i);
      if (bodyOfRoot[r] == 0xffffffffu) bodyOfRoot[r] = out.nBodies++;
      out.bodyOf[i] = bodyOfRoot[r];
    }
    out.bodyPtr.assign(out.nBodies + 1, 0);
    for (uint32_t i = 0; i < n; ++i) ++out.bodyPtr[out.bodyOf[i] + 1];
    for (uint32_t b = 0; b < out.nBodies; ++b) out.bodyPtr[b + 1] += out.bodyPtr[b];
    out.bodyNodes.assign(n, 0);
    std::vector<uint32_t> cur(out.bodyPtr.begin(), out.bodyPtr.end() - 1);
    for (uint32_t i = 0; i < n; ++i) {
      const uint32_t b = out.bodyOf[i];
      out.rankInBody[i] = cur[b] - out.bodyPtr[b];
      out.bodyNodes[cur[b]++] = i;
    }
    out.colRank.resize(out.col.size());
    for (uint32_t r = 0; r < n; ++r)
      for (int k = out.rowPtr[r]; k < out.rowPtr[r + 1]; ++k) {
        const uint32_t c = (uint32_t)out.col[k];
        out.colRank[k] = out.bodyOf[c] == out.bodyOf[r] ? out.rankInBody[c] : 0xffffffffu;
      }
  }
  buildSegments(out);
  out.blockInv.assign((size_t)out.nBlocks * 1024, 0.0f);
  auto invertBlocks = [&](unsigned t) {
    std::vector<double> a(32 * 32), inv(32 * 32);
    int slotOf[32];
    for (uint32_t b = t; b < out.nBlocks; b += T) {
      const int* nodes = &bn[32 * b];
      int m = 0;
      while (m < 32 && nodes[m] >= 0) ++m;
      std::fill(a.begin(), a.end(), 0.0);
      for (int i = 0; i < m; ++i) {
        uint32_t r = (uint32_t)nodes[i];
        for (int k = out.rowPtr[r]; k < out.rowPtr[r + 1]; ++k) {
          uint32_t c = (uint32_t)out.col[k];
          if (blockOf[c] != (int)b) continue;
          int j = 0;
          while (nodes[j] != (int)c) ++j;
          a[32 * i + j] = out.val[k];
        }
      }
      (void)slotOf;
      // Cholesky a = L L^T (in place, lower), then inverse = L^-T L^-1
      bool ok = true;
      for (int j = 0; j < m && ok; ++j) {
        double d = a[32 * j + j];
        for (int k = 0; k < j; ++k) d -= a[32 * j + k] * a[32 * j + k];
        if (!(d > 0.0)) { ok = false; break; }
        d = std::sqrt(d);
        a[32 * j + j] = d;
        for (int i = j + 1; i < m; ++i) {
          double s = a[32 * i + j];
          for (int k = 0; k < j; ++k) s -= a[32 * i + k] * a[32 * j + k];
          a[32 * i + j] = s / d;
        }
      }
      float* dst = &out.blockInv[(size_t)b * 1024];
      if (!ok) {  // not SPD (should not happen: S has M/h^2 on the diagonal): fall back to Jacobi
        for (int i = 0; i < m; ++i) {
          uint32_t r = (uint32_t)nodes[i];
          double d = 1.0;
          for (int k = out.rowPtr[r]; k < out.rowPtr[r + 1]; ++k) if ((uint32_t)out.col[k] == r) d = out.val[k];
          dst[32 * i + i] = (float)(1.0 / d);
        }
        continue;
      }
      // inv(L): forward substitution per column
      std::fill(inv.begin(), inv.end(), 0.0);
      for (int c = 0; c < m; ++c) {
        inv[32 * c + c] = 1.0 / a[32 * c + c];
        for (int i = c + 1; i < m; ++i) {
          double s = 0.0;
          for (int k = c; k < i; ++k) s -= a[32 * i + k] * inv[32 * k + c];
          inv[32 * i + c] = s / a[32 * i + i];
        }
      }
      for (int i = 0; i < m; ++i)
        for (int j = 0; j <= i; ++j) {
          double s = 0.0;
          for (int k = i; k < m; ++k) s += inv[32 * k + i] * inv[32 * k + j];
          dst[32 * i + j] = dst[32 * j + i] = (float)s;
        }
    }
  };
  {
    std::vector<std::thread> pool;
    for (unsigned t = 1; t < T; ++t) pool.emplace_back(invertBlocks, t);
    invertBlocks(0);
    for (auto& th : pool) th.join();
  }
}

}  // namespace pies
